"""Multi-stream inference latency of M-A on one GPU: one infer.MultiStreamScorer push for S streams against S infer.GraphedStreamingScorer
pushes one after another.

  python tools/multistream_latency.py [--out DIR] [--ticks K]

M-A in bf16 with zero VAE noise, uint8 240x360 frames, 16-frame windows, stride 4.  For S in {1, 8, 32, 64} streams and n in {4, 16}
frames per stream and tick, every tick is timed twice on the same frames, the two ways alternating tick by tick (and which goes first):
the wall time of one MultiStreamScorer.push plus a device synchronise, and of S GraphedStreamingScorer.push calls plus one synchronise
(what a caller waiting for every stream's scores sees).  Reported: p50 / p99 per tick, the aggregate rate in frames/s, and the largest
relative difference between the two ways' scores.  Then the multi-stream scorer runs a ragged schedule (random per-stream counts in
[0, n], one stream starting over every 50 ticks) and its graph count is reported against ceil(n / stride) + 1.  The GPU name and power
limit are read in the same run.  Writes multistream_latency.md / .json under --out (default: the current directory).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import random
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import cvad_b200  # noqa: E402,F401
from cvad_b200 import infer  # noqa: E402
from cvad_b200.ma import CausalAnomalyDetector  # noqa: E402
from stream_latency import ZeroNoise, gpu_info, pct  # noqa: E402

STREAMS = (1, 8, 32, 64)
CHUNKS = (4, 16)
T, STRIDE, H, W, CAP = 16, 4, 240, 360, 64
RAGGED_TICKS, RESET_EVERY = 200, 50


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def run(m, S, n, ticks, gen):
    multi = infer.MultiStreamScorer(m, S, clip_len=T, stride=STRIDE, capacity=CAP)
    singles = [infer.GraphedStreamingScorer(m, clip_len=T, stride=STRIDE, capacity=CAP) for _ in range(S)]
    pool = [torch.randint(0, 256, (S, n, 1, H, W), device="cuda", dtype=torch.uint8, generator=gen) for _ in range(4)]
    warm = (T + n - 1) // n + 2            # until every push completes the same number of windows: one graph key per scorer
    ways = {"multi": lambda x: [s for s, _ in multi.push(x)],
            "sequential": lambda x: [sc.push(x[k])[0] for k, sc in enumerate(singles)]}
    times = {w: [] for w in ways}
    max_rel = 0.0
    for it in range(warm + ticks):
        x = pool[it % len(pool)]
        order = ("multi", "sequential") if it % 2 == 0 else ("sequential", "multi")
        got = {}
        for w in order:
            dt, got[w] = timed(lambda: ways[w](x))
            if it >= warm:
                times[w].append(dt)
        for a, b in zip(got["multi"], got["sequential"]):
            assert a.shape == b.shape
            if b.numel():
                max_rel = max(max_rel, float((a - b).abs().max() / b.abs().max().clamp_min(1e-12)))
    row = {"streams": S, "frames_per_stream": n, "ticks": ticks, "max_rel_score_diff": max_rel,
           "steady_graphs": len(multi.graphs), "steady_keys": sorted(list(k[:2]) for k in multi.graphs)}
    for w, v in times.items():
        row[w] = {"p50_ms": 1e3 * pct(v, 50), "p99_ms": 1e3 * pct(v, 99), "frames_per_s": S * n * len(v) / sum(v)}
    row["p50_speedup"] = row["sequential"]["p50_ms"] / row["multi"]["p50_ms"]
    del singles
    # ragged schedule on the multi-stream scorer: random counts, one stream starting over every RESET_EVERY ticks
    rnd = random.Random(S * 100 + n)
    keys = {k[:2] for k in multi.graphs}
    for it in range(RAGGED_TICKS):
        if it % RESET_EVERY == RESET_EVERY - 1:
            multi.reset(rnd.randrange(S))
        counts = [rnd.randint(0, n) for _ in range(S)]
        wins = [infer.window_count(f, w, c, False, T, STRIDE)[1] for f, w, c in zip(multi.n_frames, multi.next_window, counts)]
        if any(counts):
            keys.add((n, max(wins)))
        multi.push(pool[it % len(pool)], counts)
    torch.cuda.synchronize()
    assert multi.cursors.tolist() == [[a, b] for a, b in zip(multi.n_frames, multi.next_window)]
    row["ragged"] = {"ticks": RAGGED_TICKS, "graphs": len(multi.graphs), "distinct_keys": len(keys), "bound": math.ceil(n / STRIDE) + 1}
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.getcwd(), help="directory for multistream_latency.md / .json")
    ap.add_argument("--ticks", type=int, default=200, help="timed ticks per (streams, frames per stream)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("multistream_latency.py measures on a CUDA device; none is visible")
    torch.manual_seed(0)
    m = CausalAnomalyDetector().cuda().eval().set_precision("bf16")
    m.noise = ZeroNoise()
    gen = torch.Generator(device="cuda").manual_seed(1)
    rows = []
    for n in CHUNKS:
        for S in STREAMS:
            rows.append(run(m, S, n, args.ticks, gen))
            r = rows[-1]
            print(f"S={S} n={n}: multi p50 {r['multi']['p50_ms']:.3f} ms, sequential p50 {r['sequential']['p50_ms']:.3f} ms", flush=True)
            torch.cuda.empty_cache()
    info = gpu_info()
    res = {"gpu": info, "torch": torch.__version__, "windows": {"clip_len": T, "stride": STRIDE, "H": H, "W": W, "capacity": CAP},
           "rows": rows}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "multistream_latency.json"), "w") as f:
        json.dump(res, f, indent=1)
    lines = [f"GPU (name, power limit, read in the same run): {info}", "",
             f"Wall time per tick (host clock around the pushes of one tick + one synchronize), M-A bf16, uint8 {H}x{W} frames, {T}-frame "
             f"windows, stride {STRIDE}, ring capacity {CAP}. `multi` = one `MultiStreamScorer.push` for all S streams; `sequential` = S "
             "`GraphedStreamingScorer.push` calls one after another. The two alternate tick by tick on the same frames.", "",
             "| streams S | frames / stream / tick | ticks | multi p50 ms | multi p99 ms | multi frames/s | sequential p50 ms | "
             "sequential p99 ms | sequential frames/s | p50 speed-up | max rel score diff |",
             "|---:|---:|---:|---:|---:|---:|---:|---:|---:|---:|---:|"]
    for r in rows:
        a, b = r["multi"], r["sequential"]
        lines.append(f"| {r['streams']} | {r['frames_per_stream']} | {r['ticks']} | {a['p50_ms']:.3f} | {a['p99_ms']:.3f} | "
                     f"{a['frames_per_s']:.0f} | {b['p50_ms']:.3f} | {b['p99_ms']:.3f} | {b['frames_per_s']:.0f} | "
                     f"{r['p50_speedup']:.1f}x | {r['max_rel_score_diff']:.2e} |")
    lines += ["", f"Graphs of the multi-stream scorer after a further {RAGGED_TICKS} ragged ticks (random per-stream counts in [0, n], one "
              f"stream reset every {RESET_EVERY} ticks), against the distinct (n, m) keys the run needed and the bound ceil(n / stride) + 1:",
              "", "| streams S | frames / stream / tick | graphs in steady state | graphs after the ragged run | distinct (n, m) | bound |",
              "|---:|---:|---:|---:|---:|---:|"]
    for r in rows:
        g = r["ragged"]
        lines.append(f"| {r['streams']} | {r['frames_per_stream']} | {r['steady_graphs']} | {g['graphs']} | {g['distinct_keys']} | {g['bound']} |")
    with open(os.path.join(args.out, "multistream_latency.md"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
