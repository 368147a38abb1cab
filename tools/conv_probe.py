#!/usr/bin/env python
"""Per-layer timing of the flat tensor-core convolutions at the benchmark shapes (512 frames): forward, data-gradient and
weight-gradient of the eight 3x3 layers (cad:150-153), CUDA events, L2 flushed between runs.  Development tool."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cvad_b200  # noqa: E402
from cvad_b200 import tc  # noqa: E402
from cvad_b200.ops import _call, _ptr, _st  # noqa: E402

LAYERS = [(60, 90, 32, 32, 1), (60, 90, 32, 32, 1), (60, 90, 32, 64, 2), (30, 45, 64, 64, 1), (30, 45, 64, 128, 2), (15, 23, 128, 128, 1),
          (15, 23, 128, 256, 2), (8, 12, 256, 256, 1)]


def main():
    N = int(sys.argv[1]) if len(sys.argv) > 1 else 512
    only = sys.argv[2] if len(sys.argv) > 2 else ""
    reps = int(os.environ.get("REPS", "10"))
    dev = torch.device("cuda:0")
    lib = cvad_b200.ops.L()
    if os.environ.get("CVAD_DGRAD_MODE"):
        lib.cvad_flat_dgrad_mode(int(os.environ["CVAD_DGRAD_MODE"]))
    for k in range(4):
        if os.environ.get(f"CVAD_FC_TUNE{k}"):
            lib.cvad_flat_tune(k, int(os.environ[f"CVAD_FC_TUNE{k}"]))
    flush = torch.empty(256 << 20, device=dev, dtype=torch.uint8)
    bf = torch.bfloat16
    tot = {"fwd+stats": 0.0, "fwd": 0.0, "dgrad": 0.0, "dgrad-masksum": 0.0, "wgrad-staged": 0.0, "wgrad-staged-wdot": 0.0, "wgrad": 0.0}
    for li, (H, W, Ci, Co, s) in enumerate(LAYERS):
        Ho, Wo = tc.out_hw(H, W, s)
        xin = torch.randn(tc.act_shape(N, H, W, Ci, s == 2), device=dev).to(bf)
        w = torch.randn(Co, Ci, 3, 3, device=dev) * 0.05
        b = torch.zeros(Co, device=dev)
        wf = torch.empty(9 * Co, Ci, device=dev, dtype=bf)
        wd = torch.empty(9 * Ci, Co, device=dev, dtype=bf)
        _call("cvad_flat_pack_w3x3_bf16", _ptr(w), Co, Ci, s, _ptr(wf), _ptr(wd), _st())
        y = torch.empty(N, Ho + 2, Wo + 2, Co, device=dev, dtype=bf)
        dy = torch.randn(N, Ho + 2, Wo + 2, Co, device=dev).to(bf)
        dx = torch.empty_like(xin)
        dw = torch.zeros(Co, Ci, 3, 3, device=dev)
        ws = torch.zeros(2 * Co, device=dev, dtype=torch.float64)
        ws_in = torch.zeros(4 * Ci, device=dev, dtype=torch.float64)
        mask = torch.randint(0, 256, (xin.numel() // 8,), device=dev, dtype=torch.uint8)        # the ReLU bitmask of the layer below
        scr = torch.zeros(9 * Co * Ci, device=dev)
        calls = {
            "fwd+stats": lambda: _call("cvad_flat_conv3x3_fwd_stats_bf16", _ptr(xin), _ptr(wf), _ptr(b), _ptr(y), N, H, W, Ci, Co, s, _ptr(ws), _st()),
            "fwd": lambda: _call("cvad_flat_conv3x3_fwd_bf16", _ptr(xin), _ptr(wf), _ptr(b), _ptr(y), N, H, W, Ci, Co, s, _st()),
            "dgrad": lambda: _call("cvad_flat_conv3x3_dgrad_bf16", _ptr(dy), _ptr(wd), _ptr(dx), N, H, W, Ci, Co, s, _st()),
            "dgrad-masksum": lambda: _call("cvad_flat_conv3x3_dgrad_masksum_bf16", _ptr(dy), _ptr(wd), _ptr(dx), N, H, W, Ci, Co, s, _ptr(mask),
                                           _ptr(ws_in), _st()),
            "wgrad-staged": lambda: _call("cvad_flat_conv3x3_wgrad_staged_bf16", _ptr(xin), _ptr(dy), _ptr(dw), _ptr(scr), N, H, W, Ci, Co, s, _st()),
            "wgrad-staged-wdot": lambda: _call("cvad_flat_conv3x3_wgrad_staged_wdot_bf16", _ptr(xin), _ptr(dy), _ptr(dw), _ptr(scr), N, H, W, Ci, Co,
                                               s, _ptr(w), _ptr(ws_in), _st()),
            "wgrad": lambda: _call("cvad_flat_conv3x3_wgrad_bf16", _ptr(xin), _ptr(dy), _ptr(dw), N, H, W, Ci, Co, s, _st()),
        }
        if os.environ.get("STEP_ONLY"):           # exactly the convolution launches of one train step, once each (for an ncu metrics pass)
            calls["fwd+stats"]()
            if li > 0:
                calls["dgrad"]()
            calls["wgrad-staged"]()
            torch.cuda.synchronize()
            continue
        gflop = 2.0 * N * Ho * Wo * 9 * Ci * Co / 1e9
        line = f"L{li} {H}x{W} {Ci}->{Co} s{s} ({gflop:5.1f} GFLOP): "
        for name, fn in calls.items():
            if only and only != name:
                continue
            fn()
            torch.cuda.synchronize()
            if os.environ.get("FC_DEBUG") and name in ("fwd", "dgrad"):
                dbg = torch.zeros(148 * 8 + 2, device=dev, dtype=torch.int64)
                dbg[148 * 8] = torch.iinfo(torch.int64).max
                cvad_b200.ops.L().cvad_flat_debug_buffer(dbg.data_ptr())
                fn()
                torch.cuda.synchronize()
                cvad_b200.ops.L().cvad_flat_debug_buffer(None)
                t_in, t_out = int(dbg[148 * 8]), int(dbg[148 * 8 + 1])
                d = dbg[:148 * 8].view(148, 8)
                live = d[:, 5] > 0
                m = d[live].double().mean(0)
                entry, l0, l1 = d[live, 5] - t_in, d[live, 6] - t_in, d[live, 7] - t_in
                line += (f"[{name} MMA-warp cycles/CTA: total {m[0]:.0f} wait src {m[1]:.0f} w {m[2]:.0f} acc {m[3]:.0f} items {m[4]:.1f}; "
                         f"ns from first CTA entry: last entry {int(entry.max())}, loop start mean {int(l0.double().mean())}, loop end mean "
                         f"{int(l1.double().mean())} max {int(l1.max())}, last exit {t_out - t_in}; "
                         f"SM clock in the loop {float((d[live, 0].double() / (d[live, 7] - d[live, 6]).double()).mean()) * 1e3:.0f} MHz] ")
            ms = 0.0
            for _ in range(reps):
                flush.fill_(1)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                ms += e0.elapsed_time(e1)
            ms /= reps
            tot[name] += ms
            line += f"{name} {ms * 1e3:7.1f} us {gflop / ms:7.1f} TF/s | "
        print(line, flush=True)
    print("totals (ms):", {k: round(v, 3) for k, v in tot.items()})


if __name__ == "__main__":
    main()
