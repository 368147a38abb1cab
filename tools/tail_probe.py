#!/usr/bin/env python
"""Time M-A's dense tail (everything behind the backbone) as it runs inside a captured train step.

    python tools/tail_probe.py [out_dir]

Builds MATrainer(precision="bf16") at the benchmarked shape (B = 32, T = 16) in train mode with FixedNoise and seeded features
(32, 16, 6144), captures model.tail(features) + the loss + loss.backward() into one CUDA graph and reports
  1. the replay time of that graph (CUDA events around 200 replays after 20 warm-up replays, uninstrumented);
  2. two spans of the causal branch on the main stream, from a second capture with external CUDA events around every library call
     (bench.profile_graph): forward = end of the GRU forward -> start of the loss, backward = end of the loss -> start of the GRU
     backward.  The brackets add their own cost to each of the small kernels in between, so the spans are upper bounds.
Prints one JSON line; the per-call table goes to out_dir/tail_probe_calls.md (a temporary directory by default).
"""
import json
import os
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import cvad_b200  # noqa: E402,F401
from cvad_b200 import ops  # noqa: E402
from cvad_b200.graphs import GraphedStep  # noqa: E402
from cvad_b200.ma import CausalAnomalyDetector, MATrainer  # noqa: E402
from cvad_b200.noise import FixedNoise  # noqa: E402

B, T, FEAT = 32, 16, 6144
SPANS = [("cvad_gru_fwd_f32", "cvad_ma_loss_f32", "causal branch forward (end of GRU forward -> start of loss)"),
         ("cvad_ma_loss_f32", "cvad_gru_bwd_f32", "causal branch backward (end of loss -> start of GRU backward)")]


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else None
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    tr = MATrainer(CausalAnomalyDetector(), dev, precision="bf16")
    tr.model.train()
    gen = torch.Generator().manual_seed(1)
    feats = torch.randn(B, T, FEAT, generator=gen).to(dev)
    labels = torch.randint(0, 2, (B,), generator=gen).to(dev)
    keep = lambda shape, p: (torch.rand(shape, generator=gen) >= p).float().to(dev)
    tr.model.noise = FixedNoise({"eps": torch.randn(B, 5, 6, generator=gen).to(dev), "det0": keep((B, T, 512), 0.3),
                                 "det1": keep((B, T, 256), 0.2), "scorer0": keep((B, 64), 0.2), "cls0": keep((B, 512), 0.3),
                                 "cls1": keep((B, 256), 0.2)})

    def step(f, y):
        tr.optimizer.zero_grad()
        f = f.detach().requires_grad_(True)
        out = tr.model.tail(f)
        loss, comp = tr.loss_on_device(out, y)
        with ops.param_grad_overlap():
            loss.backward()
        return (comp,)

    def make():
        gs = GraphedStep(step, (feats, labels), tr.mutated_tensors())
        return lambda: gs(feats, labels)

    replay = make()
    for _ in range(20):
        replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(200):
        replay()
    e1.record()
    torch.cuda.synchronize()
    graph_us = e0.elapsed_time(e1) / 200 * 1e3

    out_dir = out_dir or tempfile.mkdtemp()
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "tail_probe_calls.md")
    bench.profile_graph(make, path, "M-A tail graph (batch 32: tail + loss + backward)", reps=20, spans=SPANS)
    spans = {}
    for line in open(path):
        for _a, _b, label in SPANS:
            if line.startswith(label + ":"):
                spans[label] = float(line.split(":")[1].split("us")[0])
    props = torch.cuda.get_device_properties(dev)
    print(json.dumps({"device": props.name, "tail_graph_replay_us": round(graph_us, 1), "instrumented_spans_us": spans}))


if __name__ == "__main__":
    main()
