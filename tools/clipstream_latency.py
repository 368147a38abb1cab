"""Multi-stream inference latency of M-B on one GPU from raw camera frames: one infer.MultiStreamClipScorer push per tick against what a
user writes without it, and the time of the two frame-ring kernels.

  python tools/clipstream_latency.py [--out DIR] [--ticks K]

M-B with the shipped checkpoint (tests/golden/best_improved_model.pth), raw 360x640 BGR uint8 frames (Avenue's frame size) resized to
64x64, 8-frame windows at stride 4 (bbox:392).  For S in {1, 8, 64} streams and n in {4, 8} frames per stream and tick, the two ways
alternate tick by tick (and which goes first) on the same frames; each tick is the wall time of the pushes of that tick plus one device
synchronise (what a caller waiting for every stream's scores sees):
  scorer  one MultiStreamClipScorer.push for all S streams (one CUDA graph replay)
  eager   per stream: DeviceFrames(chunk).resized((64, 64)), the stream's device-side frame history, clips_f32 of the windows it completed,
          and model(clips)
Reported: p50 / p99 per tick, stream frames/s, and the largest relative difference between the two ways' scores.  Then the two kernels
of the scorer's graph, cvad_streams_frame_write_u8 and cvad_streams_clips_f32, are timed alone with CUDA events at 64 streams x 8 frames.
The GPU name and power limit are read in the same run.  Writes clipstream_latency.md / .json under --out (default: the current
directory).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import cvad_b200  # noqa: E402,F401
from cvad_b200 import infer  # noqa: E402
from cvad_b200.frames import DeviceFrames  # noqa: E402
from cvad_b200.mb import CausalAnomalyDetector  # noqa: E402
from cvad_b200.ops import _call, _ptr, _st  # noqa: E402
from stream_latency import gpu_info, pct  # noqa: E402

STREAMS = (1, 8, 64)
CHUNKS = (4, 8)
T, STRIDE, CAP = 8, 4, 32
H, W, SIZE = 360, 640, (64, 64)
KERNEL_REPS = 200


class EagerStreams:
    """The baseline: each stream's resized frames kept on the device, its completed windows gathered and scored eagerly, stream by stream."""

    def __init__(self, model, streams):
        self.model = model
        self.hist = [None] * streams          # resized frames from absolute index first[k] on
        self.first = [0] * streams
        self.frames = [0] * streams
        self.next = [0] * streams

    @torch.no_grad()
    def push(self, x):
        out = []
        for k in range(x.shape[0]):
            r = DeviceFrames(x[k], x.device).resized(SIZE).data
            h = r if self.hist[k] is None else torch.cat([self.hist[k], r])
            self.frames[k] += x.shape[1]
            done = (self.frames[k] - T) // STRIDE + 1 if self.frames[k] >= T else 0
            if done > self.next[k]:
                starts = [w * STRIDE - self.first[k] for w in range(self.next[k], done)]
                s, _, _ = self.model(DeviceFrames(h, x.device).clips_f32(starts, T))
                out.append(s.reshape(-1))
                self.next[k] = done
            else:
                out.append(torch.empty(0, device=x.device))
            drop = self.next[k] * STRIDE - self.first[k]          # frames no window needs any more
            self.hist[k], self.first[k] = h[drop:], self.first[k] + drop
        return out


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def run(m, S, n, ticks, gen):
    scorer = infer.MultiStreamClipScorer(m, S, clip_len=T, stride=STRIDE, capacity=CAP, size=SIZE)
    eager = EagerStreams(m, S)
    pool = [torch.randint(0, 256, (S, n, H, W, 3), device="cuda", dtype=torch.uint8, generator=gen) for _ in range(4)]
    warm = T // n + 2 * STRIDE                 # every graph key of the steady state is captured before timing
    ways = {"scorer": lambda x: [r[0] for r in scorer.push(x)], "eager": eager.push}
    times = {w: [] for w in ways}
    max_rel, windows = 0.0, 0
    for it in range(warm + ticks):
        x = pool[it % len(pool)]
        order = ("scorer", "eager") if it % 2 == 0 else ("eager", "scorer")
        got = {}
        for w in order:
            dt, got[w] = timed(lambda: ways[w](x))
            if it >= warm:
                times[w].append(dt)
        for a, b in zip(got["scorer"], got["eager"]):
            assert a.shape == b.shape, (a.shape, b.shape)
            if b.numel():
                windows += b.numel()
                max_rel = max(max_rel, float((a - b).abs().max() / b.abs().max().clamp_min(1e-12)))
    assert windows > 0
    row = {"streams": S, "frames_per_stream": n, "ticks": ticks, "max_rel_score_diff": max_rel, "windows_compared": windows,
           "graphs": len(scorer.graphs)}
    for w, v in times.items():
        row[w] = {"p50_ms": 1e3 * pct(v, 50), "p99_ms": 1e3 * pct(v, 99), "frames_per_s": S * n * len(v) / sum(v)}
    row["p50_speedup"] = row["eager"]["p50_ms"] / row["scorer"]["p50_ms"]
    return row


def kernel_times(S, n, gen):
    """CUDA-event time per launch of the two frame-ring kernels at S streams x n frames (every stream keeps all n and completes
    n / stride windows), averaged over KERNEL_REPS back-to-back launches after a warm-up."""
    dw, dh = SIZE
    src = torch.randint(0, 256, (S * n, H, W, 3), device="cuda", dtype=torch.uint8, generator=gen)
    rings = torch.zeros((S, CAP, dh, dw, 3), device="cuda", dtype=torch.uint8)
    cursors = torch.tensor([[64, (64 - T) // STRIDE + 1]] * S, device="cuda", dtype=torch.int64)
    push = torch.tensor([[n, 0]] * S, device="cuda", dtype=torch.int64)
    m = n // STRIDE
    clips = torch.empty((S * m, 3, T, dh, dw), device="cuda")
    calls = {
        "cvad_streams_frame_write_u8": lambda st: _call("cvad_streams_frame_write_u8", _ptr(src), S, n, H, W, 3, _ptr(rings), CAP, dh, dw, T,
                                                        STRIDE, _ptr(cursors), _ptr(push), st),
        "cvad_streams_clips_f32": lambda st: _call("cvad_streams_clips_f32", _ptr(rings), S, CAP, dh, dw, 3, T, STRIDE, m, _ptr(cursors),
                                                   _ptr(push), 1.0 / 255.0, 1, _ptr(clips), st),
    }
    written = {"cvad_streams_frame_write_u8": S * n * dh * dw * 3, "cvad_streams_clips_f32": clips.numel() * 4}
    out = {}
    for name, fn in calls.items():
        st = _st()
        for _ in range(10):
            fn(st)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(KERNEL_REPS):
            fn(st)
        b.record()
        torch.cuda.synchronize()
        us = 1e3 * a.elapsed_time(b) / KERNEL_REPS
        out[name] = {"us_per_launch": us, "bytes_written": written[name], "written_GB_per_s": written[name] / us / 1e3}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.getcwd(), help="directory for clipstream_latency.md / .json")
    ap.add_argument("--ticks", type=int, default=200, help="timed ticks per (streams, frames per stream)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("clipstream_latency.py measures on a CUDA device; none is visible")
    m = CausalAnomalyDetector()
    ck = torch.load(os.path.join(ROOT, "tests", "golden", "best_improved_model.pth"), map_location="cpu", weights_only=False)
    m.load_state_dict(ck["model_state_dict"], strict=True)
    m = m.cuda().eval()
    gen = torch.Generator(device="cuda").manual_seed(1)
    rows = []
    for n in CHUNKS:
        for S in STREAMS:
            rows.append(run(m, S, n, args.ticks, gen))
            r = rows[-1]
            print(f"S={S} n={n}: scorer p50 {r['scorer']['p50_ms']:.3f} ms, eager p50 {r['eager']['p50_ms']:.3f} ms", flush=True)
            torch.cuda.empty_cache()
    kt = kernel_times(max(STREAMS), max(CHUNKS), gen)
    info = gpu_info()
    res = {"gpu": info, "torch": torch.__version__, "model": "M-B, tests/golden/best_improved_model.pth",
           "windows": {"clip_len": T, "stride": STRIDE, "capacity": CAP, "camera": [H, W, 3], "size": list(SIZE)}, "rows": rows,
           "kernels": {"streams": max(STREAMS), "frames_per_stream": max(CHUNKS), "reps": KERNEL_REPS, **kt}}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "clipstream_latency.json"), "w") as f:
        json.dump(res, f, indent=1)
    lines = [f"GPU (name, power limit, read in the same run): {info}", "",
             f"Wall time per tick (host clock around the pushes of one tick + one synchronize), M-B with best_improved_model.pth, raw "
             f"{H}x{W} BGR uint8 frames resized to {SIZE[0]}x{SIZE[1]}, {T}-frame windows, stride {STRIDE}, ring capacity {CAP}. "
             "`scorer` = one `MultiStreamClipScorer.push` for all S streams; `eager` = per stream `DeviceFrames(chunk).resized`, a "
             "device-side frame history, `clips_f32` of the completed windows and `model(clips)`. The two alternate tick by tick on the "
             "same frames.", "",
             "| streams S | frames / stream / tick | ticks | scorer p50 ms | scorer p99 ms | scorer frames/s | eager p50 ms | eager p99 ms | "
             "eager frames/s | p50 speed-up | max rel score diff | graphs |",
             "|---:|---:|---:|---:|---:|---:|---:|---:|---:|---:|---:|---:|"]
    for r in rows:
        a, b = r["scorer"], r["eager"]
        lines.append(f"| {r['streams']} | {r['frames_per_stream']} | {r['ticks']} | {a['p50_ms']:.3f} | {a['p99_ms']:.3f} | "
                     f"{a['frames_per_s']:.0f} | {b['p50_ms']:.3f} | {b['p99_ms']:.3f} | {b['frames_per_s']:.0f} | "
                     f"{r['p50_speedup']:.1f}x | {r['max_rel_score_diff']:.2e} | {r['graphs']} |")
    lines += ["", f"The two frame-ring kernels alone (CUDA events over {KERNEL_REPS} back-to-back launches, {max(STREAMS)} streams x "
              f"{max(CHUNKS)} frames of {H}x{W}x3, {max(CHUNKS) // STRIDE} windows per stream):", "",
              "| kernel | us per launch | bytes written | written GB/s |", "|---|---:|---:|---:|"]
    for name, k in kt.items():
        lines.append(f"| `{name}` | {k['us_per_launch']:.1f} | {k['bytes_written']} | {k['written_GB_per_s']:.0f} |")
    with open(os.path.join(args.out, "clipstream_latency.md"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
