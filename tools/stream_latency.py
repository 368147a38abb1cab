"""Streaming-inference latency of M-A on one GPU: the eager ma0.StreamingWindowScorer (bf16 backbone) against infer.GraphedStreamingScorer.

  python tools/stream_latency.py [--out DIR] [--reps R]

For pushes of 4, 16, 128, 512 and 1024 uint8 240x360 frames (16-frame windows, stride 4) it reports the wall time per push (host clock
around push + device synchronise: what a caller waiting for the scores sees), p50 and p99, and the stream rate in frames/s, with the two
scorers alternating push by push in one process on the same frames.  It also reports the device time (CUDA events) of one backbone call
at 512 frames, FrozenBackbone against the eval path of tc._BackboneBF16, and the largest relative difference between the two scorers'
scores.  The GPU name and power limit are read in the same run.  Writes stream_latency.md / .json under --out (default: the current
directory).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import cvad_b200  # noqa: E402
from cvad_b200 import infer, tc  # noqa: E402
from cvad_b200.ma import CausalAnomalyDetector  # noqa: E402
from cvad_b200.ma0 import StreamingWindowScorer  # noqa: E402
from cvad_b200.noise import DeviceNoise  # noqa: E402

CHUNKS = (4, 16, 128, 512, 1024)
T, STRIDE, H, W = 16, 4, 240, 360


class ZeroNoise(DeviceNoise):
    """eps = 0 in both scorers, so that their scores can be compared window by window."""

    def normal(self, name, shape, device):
        return torch.zeros(shape, device=device)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def pct(v, p):
    v = sorted(v)
    return v[min(len(v) - 1, int(round(p / 100.0 * (len(v) - 1))))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.getcwd(), help="directory for stream_latency.md / .json")
    ap.add_argument("--reps", type=int, default=0, help="timed pushes per scorer and chunk size (default: by chunk size)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stream_latency.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    m = CausalAnomalyDetector().to(dev).eval().set_precision("bf16")
    m.noise = ZeroNoise()
    gen = torch.Generator(device=dev).manual_seed(1)
    rows, max_rel = [], 0.0
    for n in CHUNKS:
        cap = max(256, n + T + STRIDE)
        eager = StreamingWindowScorer(m, clip_len=T, stride=STRIDE, capacity=cap)
        graphed = infer.GraphedStreamingScorer(m, clip_len=T, stride=STRIDE, capacity=cap)
        frames = torch.randint(0, 256, (4 * n if n <= 128 else n, 1, H, W), device=dev, dtype=torch.uint8, generator=gen)
        chunks = [frames[i:i + n] for i in range(0, frames.shape[0], n)]
        reps = args.reps or (300 if n <= 16 else (100 if n <= 128 else 40))
        warm = max(2, (T + n - 1) // n + 2)        # until every push completes the same number of windows: one graph key
        times = {"eager": [], "graphed": []}
        for it in range(warm + reps):
            x = chunks[it % len(chunks)]
            got = {}
            for name, sc in (("eager", eager), ("graphed", graphed)):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                s, w0 = sc.push(x)
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                got[name] = (s, w0)
                if it >= warm:
                    times[name].append(dt)
            (se, we), (sg, wg) = got["eager"], got["graphed"]
            assert we == wg and se.shape == sg.shape
            if se.numel():
                max_rel = max(max_rel, float((sg - se).abs().max() / se.abs().max().clamp_min(1e-12)))
        for name in ("eager", "graphed"):
            v = times[name]
            rows.append({"scorer": name, "frames_per_push": n, "pushes": len(v), "p50_ms": 1e3 * pct(v, 50), "p99_ms": 1e3 * pct(v, 99),
                         "frames_per_s": n * len(v) / sum(v), "graphs": len(graphed.graphs) if name == "graphed" else None})
        del eager, graphed, frames, chunks
        torch.cuda.empty_cache()

    # device time of one backbone call at 512 frames (alternating blocks of events)
    x = torch.randint(0, 256, (512, 1, H, W), device=dev, dtype=torch.uint8, generator=gen)
    fz = infer.FrozenBackbone(m.backbone)
    paths = {"FrozenBackbone": lambda: fz(x), "eval _BackboneBF16": lambda: tc.backbone_forward_bf16(m.backbone, x)}
    dev_ms = {k: [] for k in paths}
    with torch.no_grad():
        for f in paths.values():
            for _ in range(3):
                f()
        for _ in range(10):
            for k, f in paths.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(10):
                    f()
                e1.record()
                e1.synchronize()
                dev_ms[k].append(e0.elapsed_time(e1) / 10)
    backbone = {k: {"median_ms": pct(v, 50), "min_ms": min(v), "max_ms": max(v)} for k, v in dev_ms.items()}

    info = gpu_info()
    res = {"gpu": info, "torch": torch.__version__, "windows": {"clip_len": T, "stride": STRIDE, "H": H, "W": W}, "pushes": rows,
           "backbone_512": backbone, "max_rel_score_diff": max_rel}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "stream_latency.json"), "w") as f:
        json.dump(res, f, indent=1)
    lines = [f"GPU (name, power limit, read in the same run): {info}", "",
             f"Wall time per push (host clock around push + synchronize), uint8 {H}x{W} frames, {T}-frame windows, stride {STRIDE}; "
             "the two scorers alternate push by push on the same frames.", "",
             "| frames / push | scorer | pushes | p50 ms | p99 ms | stream frames/s |", "|---:|---|---:|---:|---:|---:|"]
    for r in rows:
        lines.append(f"| {r['frames_per_push']} | {r['scorer']} | {r['pushes']} | {r['p50_ms']:.3f} | {r['p99_ms']:.3f} | {r['frames_per_s']:.0f} |")
    lines += ["", "Device time of one backbone call at 512 frames (CUDA events, 10 blocks of 10 calls, alternating):", "",
              "| path | median ms | min ms | max ms |", "|---|---:|---:|---:|"]
    for k, v in backbone.items():
        lines.append(f"| {k} | {v['median_ms']:.3f} | {v['min_ms']:.3f} | {v['max_ms']:.3f} |")
    lines += ["", f"Largest relative score difference, graphed vs eager scorer, over every window of the runs above: {max_rel:.2e}"]
    with open(os.path.join(args.out, "stream_latency.md"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
