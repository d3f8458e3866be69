#!/usr/bin/env python
"""bench.py — LFB frames/s of the B200-native path (MiT-EVP mit_b3_evp + SegFormer embedding head with flow,
return_features, then MS-TCN MultiStageModel_S over the extracted features).

  python bench.py --gpus N --steps K --warmup W            # our arm (torchrun for N>1, one rank per GPU, no collective on the data path)
  python bench.py --impl reference --gpus N --steps K ...   # reference arm: the reference's algorithm on the host cores (oracle port)

Workloads (`--workload`, default `auto`):
  video2300    (auto at N = 1; BASELINE.json configs[1])  a step = one synthetic Cholec80-length video (2 300 frames, 224x224) per
               GPU: LFB extraction (batches of 800; the reference driver uses 200, generate_evp_LFB.py:36) + MS-TCN over its features.
  cholec80x80  (auto at N > 1; BASELINE.json configs[2]+[3], the north-star job)  a step = the WHOLE 80-video Cholec80-shaped job
               (184 578 frames): videos LPT-sharded over the ranks (lfb.lpt_assign), every rank extracts its own videos, the
               [T_v, 2048] blocks land in video order in one page-locked shared-memory LFB array (lfb.SharedLFB — the host-side
               gather, no collective), MS-TCN over each rank's sequences, logits gathered the same way.  Strong scaling.
  native480    (`--hw 480x854`; BASELINE.json configs[4])  a step = one batch of `--batch` (64) frames at 480x854 per GPU through the
               encoder + embedding head (no MS-TCN: 64 unrelated frames are not a sequence).
Prints ONE JSON line (rank 0).  `--dump-outputs DIR` also writes what the last timed step computed (rank 0) as DIR/<name>.npy; weights
and inputs come from fixed seeds, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

FRAMES_PER_VIDEO = 2300
# Frames per forward (= micro-batch).  The reference driver uses 200 (generate_evp_LFB.py:36).  Large batches amortise weight streams and
# launches; the exact value is chosen so that the stage-3 GEMMs (M = 196 tokens x frames, 128-row tiles on 148 SMs) fill whole waves of
# the persistent grid: 1150 frames = 11.90 waves (two equal batches of a 2 300-frame video), 1159 = 11.99 waves at every stage
# (800 = 8.28 waves wasted 8 % of the last wave: measured 123.4 vs 120.8 ms per video on the same box).
BATCH = 1150
BATCH_JOB = 1159
# first batch of the end-to-end ramp-up (then doubling up to the batch size): 96 / 192 / 384 / 768 frames are 0.99 / 1.99 / 3.97 / 7.95
# waves of stage-3 tiles, so the small batches that let the kernels start early do not waste a partial wave each
RAMP_START = 96
FLOPS_PER_FRAME_REF = 16.664e9  # reference graph @224^2 with flow (SURVEY.md §8d)
FLOPS_PER_FRAME_REF_480 = 166.02e9  # @480x854 (SURVEY.md §8d)



def gemm_kernel_sha256(root):
    """sha256 of the GEMM's device + plan code (gemm_tcgen05.cu up to the extern "C" op wrappers, gemm.cuh, gemm_epi.cuh, ptx.cuh):
    recorded next to the ncu-measured traffic so that a bench run can tell whether that capture still describes the kernel it runs."""
    import hashlib, os
    d = os.path.join(root, "deep-learning-for-surgical-video-analysis_b200", "csrc")
    h = hashlib.sha256()
    src = open(os.path.join(d, "gemm_tcgen05.cu")).read()
    h.update(src.split('extern "C"')[0].encode())
    for f in ("gemm.cuh", "gemm_epi.cuh", "ptx.cuh"):
        h.update(open(os.path.join(d, f)).read().encode())
    return h.hexdigest()


DUMP_BYTES = 64 << 20   # cap on what --dump-outputs writes


def dump_outputs(out_dir, arrays, frames):
    """Writes {name: (tensor, frame axis)} as out_dir/<name>.npy in float32.  Every tensor has `frames` entries along its frame axis;
    when the set is larger than DUMP_BYTES, the same fixed, seeded sample of frames is kept in each, and frame_index.npy lists them."""
    os.makedirs(out_dir, exist_ok=True)
    per_frame = sum(t.numel() // frames * 4 for t, _ in arrays.values())
    keep = None
    if per_frame * frames > DUMP_BYTES:
        n = DUMP_BYTES // (per_frame + 8)
        keep = torch.randperm(frames, generator=torch.Generator().manual_seed(0))[:n].sort().values
        np.save(os.path.join(out_dir, "frame_index.npy"), keep.double().numpy())
    for name, (t, axis) in arrays.items():
        if keep is not None:
            t = t.index_select(axis, keep.to(t.device))
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto", "video2300", "cholec80x80", "native480"])
    ap.add_argument("--hw", default="224x224", help="frame size HxW; 480x854 selects the native480 workload")
    ap.add_argument("--frames", type=int, default=FRAMES_PER_VIDEO)
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--pool", type=int, default=2318, help="cholec80x80: frames in the per-rank synthetic input pool the videos cycle through (rounded down to a multiple of --batch)")
    ap.add_argument("--videos", type=int, default=80, help="cholec80x80: use only the first N videos (tests)")
    ap.add_argument("--micro-batch", type=int, default=int(os.environ.get("SURGVID_MICRO_BATCH", "0")), help="frames per plan inside a forward (default: = --batch)")
    ap.add_argument("--fold-head", type=int, default=int(os.environ.get("SURGVID_FOLD_HEAD", "0")))
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (float32), to compare two builds output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    a.H, a.W = (int(v) for v in a.hw.lower().split("x"))
    if a.workload == "auto":
        a.workload = "native480" if (a.H, a.W) != (224, 224) else ("video2300" if a.gpus <= 1 else "cholec80x80")
    if a.batch is None:
        a.batch = 64 if a.workload == "native480" else (BATCH_JOB if a.workload == "cholec80x80" else BATCH)
    if a.micro_batch <= 0:
        a.micro_batch = a.batch
    return a


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms; the process is started one warm-up step early (it needs
    ~0.2 s to deliver its first line) and only samples that arrive between mark_begin() and mark_end() are used."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        self.t0, self.t1 = None, None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inside = [ln for (ts, ln) in self.lines if (self.t0 is None or ts >= self.t0) and (self.t1 is None or ts <= self.t1 + 0.05)]
        if not inside:  # a very short timed region: fall back to every sample taken under the same load
            inside = [ln for (_, ln) in self.lines]
        for ln in inside:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- reference arm / cpu baseline
def cpu_port_frames_per_sec(seconds, batch=8, frames_per_video=FRAMES_PER_VIDEO, steps=None, warmup=1, H=224, W=224, with_tcn=True):
    """The reference's algorithm for this path on the host cores: oracle port (plain PyTorch fp32 restatement, pinned to the
    reference's outputs by tests/test_oracle_cpu.py), all host threads.  Sample: `batch` frames through the encoder+head with
    flow, plus (with_tcn) MS-TCN over `frames_per_video` features; frames/s = 1 / (t_enc/batch + t_tcn/frames_per_video)."""
    import surgvid_b200  # noqa: F401
    from oracle import evp_oracle, mstcn_oracle
    from surgvid_b200 import synthetic as S

    torch.set_num_threads(os.cpu_count() or 1)
    cores = torch.get_num_threads()
    sd = S.synth_state_dict(S.evp_key_shapes("mit_b3_evp"), seed=0, mode="ref_init")
    msd = S.synth_mstcn_state_dict(mode="phase")
    cfg = S.EVP_CONFIGS["mit_b3_evp"]
    x, seg, flow = S.synth_frames(batch, seed=7, H=H, W=W)
    lfb = S.synth_lfb_features(frames_per_video, seed=3).unsqueeze(0).transpose(2, 1)

    def one():
        t0 = time.perf_counter()
        evp_oracle.evp_forward(sd, cfg, x, seg, flow)
        t1 = time.perf_counter()
        if with_tcn:
            mstcn_oracle.mstcn_forward(msd, lfb)
        t2 = time.perf_counter()
        return t1 - t0, t2 - t1

    for _ in range(warmup):
        one()
    enc, tcn, n = 0.0, 0.0, 0
    t_start = time.perf_counter()
    while True:
        a, b = one()
        enc += a; tcn += b; n += 1
        if steps is not None and n >= steps:
            break
        if steps is None and time.perf_counter() - t_start >= seconds:
            break
    per_frame = enc / (n * batch) + tcn / (n * frames_per_video)
    return {"value": 1.0 / per_frame, "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": f"{n} x (oracle encoder+head fwd on {batch} frames {H}x{W} fp32 with flow" +
                      (f" + MS-TCN over {frames_per_video} features)" if with_tcn else ")") + f", {enc + tcn:.1f} s of CPU work",
            "ms_per_step": 1e3 * (enc + tcn) / n}


def workload_text(args, world):
    if args.workload == "cholec80x80":
        return (f"80-video synthetic Cholec80-shaped job (184 578 frames, 224x224; BASELINE.json configs[2]+[3]): LFB extraction (mit_b3_evp encoder + "
                f"SegFormer head with flow, return_features) LPT-sharded by video over {world} GPU(s), ordered host gather into one page-locked "
                f"shared-memory LFB array, MS-TCN MultiStageModel_S(2,8,32,2048,14) over the 80 sequences; a step = the whole job")
    if args.workload == "native480":
        return (f"mit_b3_evp encoder + SegFormer embedding head with flow at native {args.H}x{args.W}, one batch of {args.batch} frames per GPU per step "
                f"(BASELINE.json configs[4]); no MS-TCN")
    return (f"LFB extraction (mit_b3_evp encoder + SegFormer head with flow, return_features) + MS-TCN MultiStageModel_S(2,8,32,2048,14), "
            f"one {args.frames}-frame synthetic Cholec80-length video per GPU per step, 224x224 (BASELINE.json configs[1])")


def scaling_of(args):
    return "strong" if args.workload == "cholec80x80" else "weak"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # a bounded sample of the arm's workload: 8-frame encoder+head batches (at the arm's frame size) + one MS-TCN pass over a
    # 2 300-frame sequence (skipped for native480), extrapolated per frame
    r = cpu_port_frames_per_sec(0.0, steps=max(1, args.steps), warmup=max(1, args.warmup), H=args.H, W=args.W,
                                batch=8 if (args.H, args.W) == (224, 224) else 2, with_tcn=args.workload != "native480")
    line = {"impl": "reference", "metric": "lfb_frames_per_sec", "value": r["value"], "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": scaling_of(args), "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_text(args, args.gpus),
                       "arm": "reference algorithm on host cores (oracle port; /root/reference is absent on the GPU box)"},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- our arm
class Ctx:
    """Per-process state shared by the workloads."""

    def __init__(self, args):
        import torch.distributed as dist

        import surgvid_b200  # noqa: F401
        from surgvid_b200 import synthetic as S
        from surgvid_b200.models.mix_transformer_evp import mit_b3_evp
        from surgvid_b200.mstcn import MultiStageModel_S

        self.args, self.dist, self.S = args, dist, S
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise RuntimeError("bench.py (our arm) needs a CUDA device; there is no CPU fallback")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
        model = mit_b3_evp()
        model.load_state_dict(S.synth_state_dict(S.evp_key_shapes("mit_b3_evp"), seed=0, mode="ref_init"), strict=True)
        model.micro_batch, model.fold_head = args.micro_batch, bool(args.fold_head)
        self.model = model.to(self.dev).eval()
        tcn = MultiStageModel_S(2, 8, 32, 2048, 14, True)
        tcn.load_state_dict(S.synth_mstcn_state_dict(mode="phase"), strict=True)
        self.tcn = tcn.to(self.dev).eval()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, v):
        t = torch.tensor([v], device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, v):
        t = torch.tensor([v], device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def synth_device_frames(self, T, H, W, seed):
        """x ~ N(0,1); seg = Normalize(binary mask p=0.3, same in 3 channels); flow ~ 2 N(0,1)   (SURVEY.md §8d config 1), on the GPU."""
        S, dev = self.S, self.dev
        g = torch.Generator(device=dev).manual_seed(seed)
        x = torch.randn((T, 3, H, W), device=dev, generator=g)
        mask = (torch.rand((T, 1, H, W), device=dev, generator=g) > 0.7).float().expand(T, 3, H, W)
        seg = ((mask - torch.tensor(S.NORM_MEAN, device=dev).view(1, 3, 1, 1)) / torch.tensor(S.NORM_STD, device=dev).view(1, 3, 1, 1)).contiguous()
        del mask
        flow = 2.0 * torch.randn((T, 2, H, W), device=dev, generator=g)
        return x, seg, flow

    def synth_host_raw(self, T, seed):
        """What the reference's dataset class holds after JPEG decode (SURVEY.md §8f-2): uint8 250x250 frames + segmentation maps and the
        raw fp32 RAFT field, pinned."""
        g = torch.Generator().manual_seed(seed)
        fr = torch.randint(0, 256, (T, 250, 250, 3), dtype=torch.uint8, generator=g).pin_memory()
        sg = ((torch.rand((T, 250, 250, 1), generator=g) > 0.7).to(torch.uint8) * 255).expand(T, 250, 250, 3).contiguous().pin_memory()
        fl = (2.0 * torch.randn((T, 250, 250, 2), generator=g)).pin_memory()
        return fr, sg, fl

    def timed(self, step, steps, warmup):
        """W warm-up steps, then exactly K steps between CUDA events on the launching stream, barrier + synchronize on both sides,
        max over ranks; nvidia-smi clocks sampled during the timed region (rank 0).  Also returns what the last step returned."""
        sampler = ClockSampler(self.local)
        nwarm = max(3, warmup)
        for i in range(nwarm):
            if i == nwarm - 1 and self.rank == 0:
                sampler.start()
            step()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        sampler.mark_begin()
        e0.record()
        for _ in range(steps):
            out = step()
        e1.record()
        self.barrier()
        sampler.mark_end()
        ms = self.max_over_ranks(e0.elapsed_time(e1))
        clocks = sampler.stop() if self.rank == 0 else None
        return ms, clocks, nwarm, out

    def wall(self, fn):
        """Host wall-clock of fn() between barriers, max over ranks (the end-to-end legs: copies, launches and synchronisation included)."""
        self.barrier()
        t0 = time.perf_counter()
        fn()
        self.barrier()
        return self.max_over_ranks(time.perf_counter() - t0)

    def profile_classes(self, x, seg, flow, B, flops_per_frame_ref, frames_per_sec):
        """Per-kernel-class device timing (CUDA events around every launch, on the launching stream; an untimed extra pass over x) and
        the roofline object of the dominant kernel.  Rank 0 only."""
        from surgvid_b200 import _native
        peaks = measured_peaks()
        lib = _native.lib()
        model, T = self.model, x.shape[0]
        h = model._native[self.local]["handle"]
        lib.sv_evp_set_profile(h, 1)
        ncu_range = bool(os.environ.get("SURGVID_NCU_RANGE"))   # `ncu --profile-from-start off` then captures exactly this pass
        if ncu_range:
            torch.cuda.synchronize()
            torch.cuda.profiler.start()
        with torch.no_grad():
            for b0 in range(0, T, B):
                model(x[b0:min(T, b0 + B)], seg[b0:min(T, b0 + B)], flow[b0:min(T, b0 + B)], return_features=True)
            if ncu_range:
                self.tcn.forward_videos(torch.zeros((T, 2048), device=self.dev), [T])
        torch.cuda.synchronize()
        if ncu_range:
            torch.cuda.profiler.stop()
        ms_k = (ctypes.c_double * 16)()
        n_k = (ctypes.c_int64 * 16)()
        fl = ctypes.c_double(0)
        by_k = (ctypes.c_double * 16)()
        lib.sv_evp_get_profile(h, ms_k, n_k, ctypes.byref(fl), by_k)
        if os.environ.get("SURGVID_PROFILE_CSV"):
            lib.sv_evp_dump_profile(h, os.environ["SURGVID_PROFILE_CSV"].encode())
        lib.sv_evp_set_profile(h, 0)
        names = ["gemm_tcgen05", "layernorm", "im2col", "dwconv3x3_gelu", "attention", "gauss5x5", "bilinear", "token_mean", "stem_conv"]
        tot = sum(ms_k[i] for i in range(len(names)))
        # per class: device ms, launches, share, algorithmic HBM bytes (operands + results of each launch once) and the bandwidth /
        # fraction of the measured copy peak they imply (all per `T` profiled frames)
        classes = {}
        for i, nm in enumerate(names):
            gbs = by_k[i] / (ms_k[i] / 1e3) / 1e9 if ms_k[i] else None
            classes[nm] = {"ms": ms_k[i], "launches": int(n_k[i]), "share": (ms_k[i] / tot if tot else 0.0),
                           "alg_mbytes_per_frame": by_k[i] / T / 1e6, "hbm_gbs": gbs, "hbm_frac": (gbs / peaks["hbm_gbs"] if gbs else None)}
        tflops = fl.value / (ms_k[0] / 1e3) / 1e12 if ms_k[0] else 0.0
        gbs = by_k[0] / (ms_k[0] / 1e3) / 1e9 if ms_k[0] else 0.0
        traffic, traffic_src, traffic_current = None, None, None
        for rd in ("r02", "r01"):
            tpath = os.path.join(ROOT, "profiles", rd, "gemm_traffic.json")
            if os.path.exists(tpath) and (args_hw(self.args) == (224, 224)):
                tj = json.load(open(tpath))
                # ncu measured the DRAM bytes of the GEMM launches of one micro-batch of `frames_profiled` frames; per launch of THIS run
                # (same 197 launches per micro-batch, more frames each) = bytes per frame x frames of this pass / launches of this pass
                if tj.get("traffic_bytes_per_frame"):
                    traffic = tj["traffic_bytes_per_frame"] * T / max(1, n_k[0])
                else:
                    traffic = tj.get("traffic_bytes_per_launch")
                traffic_src = tj.get("source")
                traffic_current = (tj.get("gemm_kernel_sha256") == gemm_kernel_sha256(ROOT)) if tj.get("gemm_kernel_sha256") else None
                break
        # The dominant kernel is the tcgen05 GEMM.  Its launches have an aggregate arithmetic intensity of ~130 FLOP/B (K = 64..320 for most
        # of them) against a ridge of ~213 FLOP/B, so the BINDING roofline is HBM; the tensor-pipe figures are reported alongside.
        roofline = {"bound": "hbm", "kernel": "gemm_bf16_tcgen05_kernel", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": gbs / peaks["hbm_gbs"], "traffic": traffic, "traffic_source": traffic_src,
                    # True: the GEMM device + plan code of this tree is byte-identical to the one the ncu capture was taken with
                    "traffic_capture_matches_kernel": traffic_current,
                    "peak_source": peaks["source"] + " (copy bandwidth)",
                    "avg_launch_ms": ms_k[0] / max(1, n_k[0]), "launches_profiled": int(n_k[0]), "frames_profiled": T,
                    "algorithmic_bytes_per_launch": by_k[0] / max(1, n_k[0]), "algorithmic_bytes_per_frame": by_k[0] / T,
                    "share_of_step_device_time": classes["gemm_tcgen05"]["share"],
                    "tensor": {"achieved": tflops, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                               "frac": tflops / peaks["bf16_tflops_sustained"], "algorithmic_flops_profiled": fl.value,
                               "executed_gemm_flops_per_frame": fl.value / T,
                               "peak_note": "sustained cuBLAS bf16 figure of MEASURED_PEAKS.json (kernel timed inside a long step)"}}
        whole = {"ref_graph_flops_per_frame": flops_per_frame_ref, "achieved_tflops_ref_graph": frames_per_sec / self.world * flops_per_frame_ref / 1e12,
                 "frac_of_sustained_peak": frames_per_sec / self.world * flops_per_frame_ref / 1e12 / peaks["bf16_tflops_sustained"]}
        return roofline, classes, whole

    def emit(self, line):
        if self.rank == 0:
            print(json.dumps(line), flush=True)
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def args_hw(args):
    return (args.H, args.W)


def base_line(ctx, value, ms_total, nwarm, clocks, launches, e2e, roofline, cpu, classes, whole, extra_cfg):
    a = ctx.args
    cfg = {"workload": workload_text(a, ctx.world), "batch": a.batch, "micro_batch": a.micro_batch, "fold_head": int(a.fold_head),
           "weights": "random init (reference distributions), seed 0", "parallelism": f"{ctx.world} x independent video shards, no collective on the data path"}
    cfg.update(extra_cfg)
    return {"metric": "lfb_frames_per_sec", "value": value, "unit": "frames/s", "n_gpus": ctx.world, "steps": a.steps, "warmup": nwarm,
            "ms_per_step": ms_total / a.steps, "higher_is_better": True, "scaling": scaling_of(a), "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": cfg, "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline, "cpu_baseline": cpu, "kernel_classes": classes, "tensor_roofline_whole_path": whole}


def run_video(ctx):
    """video2300 (N=1 default, weak scaling) and native480."""
    from surgvid_b200 import lfb
    a, dev, model, tcn, world, rank = ctx.args, ctx.dev, ctx.model, ctx.tcn, ctx.world, ctx.rank
    native = a.workload == "native480"
    T, B, H, W = (a.batch if native else a.frames), a.batch, a.H, a.W
    # synthetic video resident in HBM (3.7 GB fp32 per rank at 2 300 x 224^2; 0.84 GB at 64 x 480x854), far larger than the 126 MB L2
    x, seg, flow = ctx.synth_device_frames(T, H, W, 1234 + rank)
    feats = torch.empty((T, 2048), dtype=torch.float32, device=dev)
    launches = {"n": 0}

    @torch.no_grad()
    def step():
        n = 0
        for b0 in range(0, T, B):
            b1 = min(T, b0 + B)
            feats[b0:b1] = model(x[b0:b1], seg[b0:b1], flow[b0:b1], return_features=True)
            n += model.last_launch_count(dev)
        if native:
            launches["n"] = n
            return feats
        logits = tcn.forward_videos(feats, [T])
        launches["n"] = n + tcn.last_launch_count(dev)
        return logits

    ms_total, clocks, nwarm, out = ctx.timed(step, a.steps, a.warmup)
    value = world * T * a.steps / (ms_total / 1e3)
    if a.dump_outputs and rank == 0:
        # features [T, 2048]; video2300 adds the MS-TCN logits [stages, classes, T]
        dump_outputs(a.dump_outputs, {"features": (feats, 0)} if native else {"features": (feats, 0), "logits": (out, 2)}, T)

    # ---- end-to-end through the public API with HOST buffers (pinned), H2D + D2H inside the timed region
    e2e = None
    numa_cpus = lfb.bind_to_gpu_numa_node(ctx.local) if world > 1 else None   # pinned staging memory on the GPU's own NUMA node
    if not a.no_e2e:
        xh, sh, fh = x.cpu().pin_memory(), seg.cpu().pin_memory(), flow.cpu().pin_memory()
        ext = lfb.LFBExtractor(model, batch_size=B, device=dev, ramp_start=RAMP_START if B >= 4 * RAMP_START and (H, W) == (224, 224) else None)
        k = max(1, min(a.steps, 3))
        outs_h = [torch.empty((T, 2048), dtype=torch.float32).pin_memory() for _ in range(k)]
        feats_d = torch.empty((k * T, 2048), dtype=torch.float32, device=dev)
        logits_h = torch.empty((2, 14, T * k), dtype=torch.float32).pin_memory()

        @torch.no_grad()
        def e2e_run(k, raw=None):
            # k steps = k videos through the driver-level call: one pipelined pass (H2D of every batch from pinned host memory, forward,
            # D2H of the features), then MS-TCN over the k feature sequences (kept on the GPU) and D2H of the phase logits
            douts = [feats_d[i * T:(i + 1) * T] for i in range(k)]
            if raw is None:
                ext.extract_videos([(xh, sh, fh)] * k, outs=outs_h[:k], device_outs=douts)
            else:
                ext.extract_raw_videos([raw] * k, outs=outs_h[:k], device_outs=douts)
            if not native:
                lg = tcn.forward_videos(feats_d[:k * T], [T] * k)
                logits_h[:, :, :T * k].copy_(lg, non_blocking=True)
            torch.cuda.synchronize()

        e2e_run(1)
        dt = ctx.wall(lambda: e2e_run(k))
        fp32_leg = {"value": world * T * k / dt, "unit": "frames/s",
                    "h2d_bytes_per_step": int(ext.h2d_bytes // k), "d2h_bytes_per_step": int(ext.d2h_bytes // k + (0 if native else 2 * 14 * T * 4)),
                    "steps": k, "input_format": f"fp32 [T,3|3|2,{H},{W}] tensors as model_LFB receives them",
                    "api": "LFBExtractor.extract_videos(model=mit_b3_evp drop-in; the timed steps are videos of ONE pipelined call)" +
                           ("" if native else " + MultiStageModel_S.forward_videos")}
        del xh, sh, fh
        if native:
            e2e = fp32_leg
        else:
            # The headline e2e starts from what the reference's dataset class holds after JPEG decode (SURVEY.md 8f-2): uint8 250x250 frames and
            # segmentation maps + the raw fp32 RAFT field (0.88 MB/frame); Resize/CenterCrop/ToTensor/Normalize and the flow resize run on the
            # GPU.  The same chain from the fp32 tensors model_LFB receives (1.6 MB/frame) is reported beside it.
            raw = ctx.synth_host_raw(T, 11 + rank)
            e2e_run(1, raw)
            dt = ctx.wall(lambda: e2e_run(k, raw))
            e2e = {"value": world * T * k / dt, "unit": "frames/s", "h2d_bytes_per_step": int(ext.h2d_bytes // k),
                   "d2h_bytes_per_step": int(ext.d2h_bytes // k + 2 * 14 * T * 4), "steps": k,
                   "input_format": "uint8 [T,250,250,3] frames + segmentation maps and fp32 [T,250,250,2] RAFT flow (what the reference's dataset class "
                                   "holds after decode); Resize/CenterCrop/ToTensor/Normalize + flow resize on the GPU",
                   "api": "LFBExtractor.extract_raw_videos(one pipelined call; the timed steps are its videos) + MultiStageModel_S.forward_videos",
                   "from_fp32_tensors": fp32_leg}
            del raw
        e2e["host_cores_bound"] = len(numa_cpus) if numa_cpus else None

    roofline = classes = whole = None
    if rank == 0 and not a.no_profile:
        roofline, classes, whole = ctx.profile_classes(x, seg, flow, B, FLOPS_PER_FRAME_REF_480 if native else FLOPS_PER_FRAME_REF, value)
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        cpu = cpu_port_frames_per_sec(a.cpu_seconds, H=H, W=W, batch=8 if not native else 2, with_tcn=not native)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
    launches_all = ctx.sum_over_ranks(launches["n"]) * a.steps
    ctx.emit(base_line(ctx, value, ms_total, nwarm, clocks, launches_all, e2e, roofline, cpu, classes, whole,
                       {"frames_per_step_per_gpu": T, "l2": f"inputs ({x.numel() * 4 * 8 // 3 / 1e9:.1f} GB fp32 per GPU) are far larger than the 126 MB L2; no flush needed"}))


def run_cholec80(ctx):
    """The north-star job: 80 Cholec80-shaped videos, LPT-sharded by video, ordered host gather, MS-TCN (strong scaling)."""
    from surgvid_b200 import lfb
    a, dev, model, tcn, world, rank, S = ctx.args, ctx.dev, ctx.model, ctx.tcn, ctx.world, ctx.rank, ctx.S
    lengths = [int(n) for n in S.cholec80_video_lengths()[:a.videos]]
    total = sum(lengths)
    assign = lfb.lpt_assign(lengths, world)
    mine = assign[rank]
    my_len = [lengths[v] for v in mine]
    R = sum(my_len)
    B, P = a.batch, max(a.batch, (a.pool // a.batch) * a.batch)
    loads = [sum(lengths[v] for v in vs) for vs in assign]
    # Inputs: 184 578 frames are 295 GB as fp32 tensors, more than fits next to the workspace at N <= 2, so every rank keeps a POOL of P
    # distinct synthetic frames resident (3.7 GB, >> L2) and its videos cycle through it; frame t of the rank's stream is pool row t % P.
    x, seg, flow = ctx.synth_device_frames(P, a.H, a.W, 1234 + rank)
    feats_d = torch.empty((R, 2048), dtype=torch.float32, device=dev)
    douts, o = [], 0
    for T in my_len:
        douts.append(feats_d[o:o + T])
        o += T
    tag = f"{os.environ.get('MASTER_PORT', '0')}_{os.getppid() if world > 1 else os.getpid()}"
    names = (f"surgvid_lfb_{tag}", f"surgvid_logits_{tag}")
    if rank == 0:
        shared = lfb.SharedLFB(names[0], lengths, 2048, create=True)
        shared_lg = lfb.SharedLFB(names[1], lengths, 2 * 14, create=True)
    ctx.barrier()
    if rank != 0:
        shared = lfb.SharedLFB(names[0], lengths, 2048)
        shared_lg = lfb.SharedLFB(names[1], lengths, 2 * 14)
    houts, hlg = shared.blocks(mine), shared_lg.blocks(mine)
    side = torch.cuda.Stream(dev)
    ev = torch.cuda.Event()
    launches = {"n": 0}
    batches = lfb.pack_batches(my_len, B)   # (video, first frame, count) segments; batches cross video boundaries

    @torch.no_grad()
    def tcn_and_gather():
        lg = tcn.forward_videos(feats_d, my_len)                 # [2, 14, R] channel-major
        lgt = lg.permute(2, 0, 1).reshape(R, 28).contiguous()     # time-major rows for the per-video host blocks
        o = 0
        for blk, T in zip(hlg, my_len):
            blk.copy_(lgt[o:o + T], non_blocking=True)
            o += T
        return tcn.last_launch_count(dev)

    @torch.no_grad()
    def step():
        cur = torch.cuda.current_stream(dev)
        n, pos = 0, 0
        for segs in batches:
            m = sum(s[2] for s in segs)
            p0 = pos % P                                          # B divides P: a batch never wraps
            f = model(x[p0:p0 + m], seg[p0:p0 + m], flow[p0:p0 + m], return_features=True)
            n += model.last_launch_count(dev)
            feats_d[pos:pos + m] = f
            ev.record(cur)
            side.wait_event(ev)
            with torch.cuda.stream(side):                         # feature blocks -> their rows of the shared LFB, off the compute stream
                oo = pos
                for (vi, b0, k) in segs:
                    houts[vi][b0:b0 + k].copy_(feats_d[oo:oo + k], non_blocking=True)
                    oo += k
            pos += m
        n += tcn_and_gather()
        cur.wait_stream(side)                                     # the step ends when the last block is gathered
        launches["n"] = n

    ms_total, clocks, nwarm, _ = ctx.timed(step, a.steps, a.warmup)
    value = total * a.steps / (ms_total / 1e3)
    if a.dump_outputs and rank == 0:
        # the gathered arrays every rank's blocks landed in, rows in video order: features [total, 2048], logits [total, stages x classes]
        dump_outputs(a.dump_outputs, {"features": (shared.array, 0), "logits": (shared_lg.array, 0)}, total)

    e2e = None
    numa_cpus = lfb.bind_to_gpu_numa_node(ctx.local) if world > 1 else None
    if not a.no_e2e:
        ext = lfb.LFBExtractor(model, batch_size=B, device=dev, ramp_start=RAMP_START if B >= 4 * RAMP_START else None)
        k = 1 if world == 1 else max(1, min(a.steps, 2))

        @torch.no_grad()
        def job(videos, raw):
            (ext.extract_raw_videos if raw else ext.extract_videos)(videos, outs=houts, device_outs=douts)
            tcn_and_gather()
            torch.cuda.synchronize()

        def leg(videos, raw, warm_videos):
            job_w = lambda: [job(videos, raw) for _ in range(k)]   # noqa: E731
            (ext.extract_raw_videos if raw else ext.extract_videos)(warm_videos)   # allocate staging, warm the pipeline
            dt = ctx.wall(job_w)
            return {"value": total * k / dt, "unit": "frames/s", "h2d_bytes_per_step": int(ctx.sum_over_ranks(ext.h2d_bytes)),
                    "d2h_bytes_per_step": int(ctx.sum_over_ranks(ext.d2h_bytes + R * 28 * 4)), "steps": k}

        # (1) from what the reference's dataset class holds after JPEG decode (uint8 250x250 frames + segmaps, raw fp32 flow; 0.88 MB/frame,
        #     transforms on the GPU): the headline e2e.  (2) from the fp32 tensors model_LFB receives (1.6 MB/frame), reported beside it.
        Ph = P
        fr, sg, fl = ctx.synth_host_raw(Ph, 11 + rank)
        off = np.cumsum([0] + my_len)
        vids = [(lfb.CyclicFrames(fr, off[i], T), lfb.CyclicFrames(sg, off[i], T), lfb.CyclicFrames(fl, off[i], T)) for i, T in enumerate(my_len)]
        e2e = leg(vids, True, [(fr[:2 * B], sg[:2 * B], fl[:2 * B])])
        e2e.update({"host_cores_bound": (len(numa_cpus) if numa_cpus else None),
                    "input_format": "uint8 [T,250,250,3] frames + segmentation maps and fp32 [T,250,250,2] RAFT flow (what the reference's dataset "
                                    "class holds after decode); Resize/CenterCrop/ToTensor/Normalize + flow resize on the GPU",
                    "api": "LFBExtractor.extract_raw_videos(rank's videos -> rows of lfb.SharedLFB) + MultiStageModel_S.forward_videos; wall-clock "
                           "from first launch to last block gathered, max over ranks"})
        del fr, sg, fl, vids
        xh, sh, fh = x.cpu().pin_memory(), seg.cpu().pin_memory(), flow.cpu().pin_memory()
        vids = [(lfb.CyclicFrames(xh, off[i], T), lfb.CyclicFrames(sh, off[i], T), lfb.CyclicFrames(fh, off[i], T)) for i, T in enumerate(my_len)]
        e2e["from_fp32_tensors"] = leg(vids, False, [(xh[:2 * B], sh[:2 * B], fh[:2 * B])])
        e2e["from_fp32_tensors"]["api"] = "LFBExtractor.extract_videos(fp32 [T,3|3|2,224,224] pinned host tensors) + MultiStageModel_S.forward_videos"
        del xh, sh, fh, vids

    roofline = classes = whole = None
    if rank == 0 and not a.no_profile:
        roofline, classes, whole = ctx.profile_classes(x, seg, flow, B, FLOPS_PER_FRAME_REF, value)
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        cpu = cpu_port_frames_per_sec(a.cpu_seconds)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
    launches_all = ctx.sum_over_ranks(launches["n"]) * a.steps
    # order check of the gathered array (cheap, after timing): every rank's last video block is where the consumers will look for it
    ok = bool(torch.equal(houts[-1], feats_d[R - my_len[-1]:].cpu()))
    ok = ctx.sum_over_ranks(0.0 if ok else 1.0) == 0.0
    extra = {"frames_per_step": total, "videos": len(lengths), "lpt_frames_per_rank": loads, "lpt_imbalance": max(loads) / (total / world) - 1.0,
             "input_pool_frames_per_rank": P, "gather": f"page-locked shared-memory LFB array ({'pinned' if shared.pinned else 'NOT pinned'}), rows in video order",
             "gather_verified": ok,
             "l2": "the 3.7 GB resident input pool and the 16 GB workspace are far larger than the 126 MB L2; no flush needed"}
    line = base_line(ctx, value, ms_total, nwarm, clocks, launches_all, e2e, roofline, cpu, classes, whole, extra)
    shared.unlink(), shared_lg.unlink()
    ctx.emit(line)


def run_ours(args):
    ctx = Ctx(args)
    if args.workload == "cholec80x80":
        run_cholec80(ctx)
    else:
        run_video(ctx)


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
