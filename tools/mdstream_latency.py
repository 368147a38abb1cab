"""Multi-stream inference latency of M-D on one GPU: one infer.MultiStreamAutoEncoderScorer push per tick against what a user does without
it.

  python tools/mdstream_latency.py [--out DIR] [--ticks K]

M-D (md.VideoAutoEncoder, seeded default initialisation, memory bank filled with 100 rows so the memory term is live), fp32 64x64 frames in
[0.001, 0.999], 8-frame windows at stride 4, ring capacity 32.  For S x n in {1x4, 8x4, 64x4, 8x16, 64x16} (S streams, n frames per stream
and tick) the two ways alternate tick by tick (and which goes first) on the same frames; each tick is the wall time of that tick's work
plus one device synchronise (what a caller waiting for every stream's scores sees):
  scorer  one MultiStreamAutoEncoderScorer.push for all S streams (one CUDA graph replay; every frame encoded once)
  eager   every window completed that tick cut as a clip from its stream's device-side frames, all of them scored in one batch by
          md.calculate_anomaly_scores (every window encodes all of its frames)
Reported: p50 / p99 per tick, stream frames/s, and the largest relative difference between the two ways' scores.  The GPU name and power
limit are read in the same run.  Writes mdstream_latency.md / .json under --out (default: the current directory).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import cvad_b200  # noqa: E402,F401
from cvad_b200 import infer, md  # noqa: E402
from stream_latency import gpu_info, pct  # noqa: E402

CONFIGS = ((1, 4), (8, 4), (64, 4), (8, 16), (64, 16))
T, STRIDE, CAP = 8, 4, 32


class EagerStreams:
    """The baseline: each stream's frames kept on the device; every window completed in a tick is cut from them and all of the tick's
    windows are scored in one calculate_anomaly_scores batch."""

    def __init__(self, model, streams):
        self.model = model
        self.hist = [None] * streams          # frames from absolute index first[k] on
        self.first = [0] * streams
        self.frames = [0] * streams
        self.next = [0] * streams

    @torch.no_grad()
    def push(self, x):
        clips, per_stream = [], []
        for k in range(x.shape[0]):
            h = x[k] if self.hist[k] is None else torch.cat([self.hist[k], x[k]])
            self.frames[k] += x.shape[1]
            done = (self.frames[k] - T) // STRIDE + 1 if self.frames[k] >= T else 0
            clips += [h[w * STRIDE - self.first[k]:w * STRIDE - self.first[k] + T] for w in range(self.next[k], done)]
            per_stream.append(done - self.next[k])
            self.next[k] = done
            drop = self.next[k] * STRIDE - self.first[k]          # frames no window needs any more
            self.hist[k], self.first[k] = h[drop:], self.first[k] + drop
        if not clips:
            return [np.zeros(0, dtype=np.float32)] * len(per_stream)
        scores, _, _, _ = md.calculate_anomaly_scores(self.model, [(torch.stack(clips), np.zeros(len(clips)))], device=x.device)
        return np.split(scores, np.cumsum(per_stream)[:-1])


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def run(m, S, n, ticks, gen):
    scorer = infer.MultiStreamAutoEncoderScorer(m, S, clip_len=T, stride=STRIDE, capacity=CAP)
    eager = EagerStreams(m, S)
    pool = [torch.rand((S, n, 1, 64, 64), device="cuda", generator=gen) * 0.998 + 0.001 for _ in range(4)]
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
            a = a.cpu().numpy()
            assert a.shape == b.shape, (a.shape, b.shape)
            if b.size:
                windows += b.size
                max_rel = max(max_rel, float(np.abs(a.astype(np.float64) - b).max() / max(np.abs(b).max(), 1e-12)))
    assert windows > 0
    row = {"streams": S, "frames_per_stream": n, "ticks": ticks, "max_rel_score_diff": max_rel, "windows_compared": windows,
           "graphs": len(scorer.graphs)}
    for w, v in times.items():
        row[w] = {"p50_ms": 1e3 * pct(v, 50), "p99_ms": 1e3 * pct(v, 99), "frames_per_s": S * n * len(v) / sum(v)}
    row["p50_speedup"] = row["eager"]["p50_ms"] / row["scorer"]["p50_ms"]
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.getcwd(), help="directory for mdstream_latency.md / .json")
    ap.add_argument("--ticks", type=int, default=200, help="timed ticks per (streams, frames per stream)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mdstream_latency.py measures on a CUDA device; none is visible")
    torch.manual_seed(0)
    m = md.VideoAutoEncoder().cuda().eval()
    m.update_memory(torch.randn(100, 64, device="cuda"))
    gen = torch.Generator(device="cuda").manual_seed(1)
    rows = []
    for S, n in CONFIGS:
        rows.append(run(m, S, n, args.ticks, gen))
        r = rows[-1]
        print(f"S={S} n={n}: scorer p50 {r['scorer']['p50_ms']:.3f} ms, eager p50 {r['eager']['p50_ms']:.3f} ms", flush=True)
        torch.cuda.empty_cache()
    info = gpu_info()
    res = {"gpu": info, "torch": torch.__version__, "model": "M-D, seeded default initialisation, 100 memory rows",
           "windows": {"clip_len": T, "stride": STRIDE, "capacity": CAP, "frame": [1, 64, 64]}, "rows": rows}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "mdstream_latency.json"), "w") as f:
        json.dump(res, f, indent=1)
    lines = [f"GPU (name, power limit, read in the same run): {info}", "",
             f"Wall time per tick (host clock around one tick's work + one synchronize), M-D, fp32 64x64 frames, {T}-frame windows, stride "
             f"{STRIDE}, ring capacity {CAP}. `scorer` = one `MultiStreamAutoEncoderScorer.push` for all S streams (every frame encoded "
             "once); `eager` = every window completed that tick cut from its stream's device-side frames and scored in one "
             "`md.calculate_anomaly_scores` batch (every window encodes its frames). The two alternate tick by tick on the same frames.", "",
             "| streams S | frames / stream / tick | ticks | scorer p50 ms | scorer p99 ms | scorer frames/s | eager p50 ms | eager p99 ms | "
             "eager frames/s | p50 speed-up | max rel score diff | graphs |",
             "|---:|---:|---:|---:|---:|---:|---:|---:|---:|---:|---:|---:|"]
    for r in rows:
        a, b = r["scorer"], r["eager"]
        lines.append(f"| {r['streams']} | {r['frames_per_stream']} | {r['ticks']} | {a['p50_ms']:.3f} | {a['p99_ms']:.3f} | "
                     f"{a['frames_per_s']:.0f} | {b['p50_ms']:.3f} | {b['p99_ms']:.3f} | {b['frames_per_s']:.0f} | "
                     f"{r['p50_speedup']:.2f}x | {r['max_rel_score_diff']:.2e} | {r['graphs']} |")
    with open(os.path.join(args.out, "mdstream_latency.md"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
