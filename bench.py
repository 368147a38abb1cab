#!/usr/bin/env python
"""Benchmarks of the hot path on synthetic Avenue-shaped clips (BASELINE.json configs).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--batch B] [--frames u8|f32]
                    [--dump-outputs DIR]

Workloads (``--workload``; the default is the headline, BASELINE.json configs[1]):
  ma_train    C2  M-A (causal_anomaly_detection.py) training step, 32 clips x 16 frames x 240x360 per GPU, bf16 operands  [clips/s]
  mc_infer    C1  M-C (minicausal_vad_complete3.py) inference, (4,1,16,64,64) per GPU                                     [frames/s]
  mb_train    C3  M-B (avenue_training_script1/2.py loop body) training step from the shipped checkpoint, per-GPU batch 32 [clips/s]
  me_windows  C4  bbox sliding windows: 298 stride-4 windows of a 1200-frame video as batches (vs the batch-1 loop)        [clips/s]
  mc_long     C5  long-sequence inference sweep T = 64 / 128 / 256, 4 clips per GPU per T                                  [frames/s]

One JSON line on stdout (rank 0).  A "step" is one pass of the hot path over one batch.
  value         units/s with the inputs resident in HBM (M-A: the batch exceeds the 126 MB L2, so every step streams it; the small models:
                an L2 flush is NOT needed to be honest about them -- they are launch/latency bound, config.l2 says which applies)
  e2e           the same through the public API with the batch in PINNED HOST memory: H2D copy of the step's inputs and a D2H read of the
                step's result inside the timed region
  roofline      the dominant kernel family timed with CUDA events inside the replayed step, against MEASURED_PEAKS.json
  cpu_baseline  the reference's own code (oracle/_ref, kind "reference") or its oracle port (kind "port") on the host cores, bounded sample
  self_check    (ma_train, mc_infer, mb_train) the first step's result against the committed golden fixture made by the unmodified reference

--dump-outputs DIR writes what the last timed step returned (rank 0) as DIR/<name>.npy: every input and initial state is seeded, so two
builds run with the same arguments can be compared output for output.  ma_train / mb_train: loss_components and the parameter arena
after the step (M-A also its anomaly_scores); mc_infer / mc_long: scores_T<T> per sequence length; me_windows: scores, adjacency, features.
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

T, H, W = 16, 240, 360
PER_GPU_BATCH = 32
# algorithmic FLOPs (2*MAC) per frame of the eight 3x3 convolutions (SURVEY.md 8d): forward, and forward+dgrad+wgrad
CONV_FWD_MFLOP = [99.53, 99.53, 49.77, 99.53, 50.87, 101.74, 56.62, 113.25]
CONV_TRAIN_MFLOP = sum(CONV_FWD_MFLOP) * 3 - CONV_FWD_MFLOP[0]      # layer1.0 needs no data-gradient (frozen stem below it)
# compulsory HBM bytes of the same 23 calls for 512 frames: every operand read once and every result written once in bf16 over the
# logical (unpadded) tensors; weights and weight-gradients are negligible.  (elements per frame of each layer's input / output)
_CONV_IO = [(172800, 172800), (172800, 172800), (172800, 86400), (86400, 86400), (86400, 44160), (44160, 44160), (44160, 24576), (24576, 24576)]
CONV_ALG_BYTES = sum(2 * 512 * ((i + o) + (i + o) + ((i + o) if k else 0)) for k, (i, o) in enumerate(_CONV_IO))

WORKLOADS = {
    "ma_train": ("train clips/sec", "clips/s", "M-A (causal_anomaly_detection.py) train step, synthetic Avenue clips (32,16,1,240,360) per GPU"),
    "mc_infer": ("inference frames/sec", "frames/s", "M-C (minicausal_vad_complete3.py) inference, synthetic clips (4,1,16,64,64) per GPU"),
    "mb_train": ("train clips/sec", "clips/s", "M-B (avenue_training_script1/2.py loop body) train step from best_improved_model.pth, (B,3,8,64,64) per GPU"),
    "me_windows": ("inference clips/sec", "clips/s", "bbox sliding windows: 298 stride-4 windows (1,3,8,64,64) of one 1200-frame video per GPU, batched"),
    "mc_long": ("inference frames/sec", "frames/s", "M-C long-sequence inference sweep, (4,1,T,64,64) for T in 64/128/256 per GPU"),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1341.2), d.get("hbm_gbs", 6499.0), "measured"
    return 1400.0, 6650.0, "fallback"


def conv_family_traffic():
    """DRAM bytes the convolution family moves per 512-frame step, from the committed ncu capture (tools/conv_traffic.py)."""
    p = os.path.join(ROOT, "profiles", "conv_family_traffic.json")
    if not os.path.exists(p):
        return None, None
    d = json.load(open(p))
    return d.get("bytes_per_step"), d.get("source")


_T0 = time.time()


def trace(msg):
    """Stage markers on stderr (CVAD_BENCH_TRACE=1): where every rank is, should a multi-GPU run stall."""
    if os.environ.get("CVAD_BENCH_TRACE", "0") == "1":
        print(f"[bench rank {os.environ.get('RANK', '0')} +{time.time() - _T0:6.1f}s] {msg}", file=sys.stderr, flush=True)


class ClockSampler(threading.Thread):
    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        mhz = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples if len(s) > 2 + i)]
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None, "sm_max_mhz": int(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                "reasons": reasons}


def synth_batch(B, seed, frames="f32"):
    """The M-A batch of one rank: raw 0..255 grayscale frames; ``f32`` = after the reference's host-side Normalize (cad:1177-1179), ``u8`` =
    the raw bytes (normalised on the device, bit-identical result).  Labels: bernoulli(0.3)."""
    import synth
    x = synth.ma_clips(B, T, H, W, seed, wide=True)
    if frames == "u8":
        x = (x * 0.5 + 0.5).round().to(torch.uint8)       # exact inverse of (v - 0.5) / 0.5 for integer v
    y = (torch.rand(B, generator=synth.gen(seed + 9)) < 0.3).long()
    return x, y


def ma_noise_for(B, xseed):
    import synth
    eps = torch.randn(B, 5, 6, generator=synth.gen(xseed + 1))
    keep = {"det0": synth.keep_mask((B, T, 512), 0.3, xseed + 2), "det1": synth.keep_mask((B, T, 256), 0.2, xseed + 3),
            "scorer0": synth.keep_mask((B, 64), 0.2, xseed + 4), "cls0": synth.keep_mask((B, 512), 0.3, xseed + 5),
            "cls1": synth.keep_mask((B, 256), 0.2, xseed + 6)}
    return eps, keep


def gold(name):
    import synth
    return synth.golden(name)


DUMP_LIMIT_BYTES = 64 * 10**6


def dump_outputs(path, arrays):
    """``--dump-outputs``: one ``<name>.npy`` per array, float64 kept, everything else written as float32."""
    import numpy as np
    host = {k: v.detach().cpu().to(torch.float64 if v.dtype == torch.float64 else torch.float32) for k, v in arrays.items()}
    total = sum(t.numel() * t.element_size() for t in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(path, exist_ok=True)
    for k, t in host.items():
        np.save(os.path.join(path, k + ".npy"), t.numpy())


# ============================================================================================ the reference's CPU arm
def _ref_module(name):
    """The UNMODIFIED reference script ``name`` from oracle/_ref (or /root/reference in the build container); None when absent."""
    from oracle import ref_harness
    d = ref_harness.reference_dir()
    if d is None:
        return None
    return ref_harness.import_ref(name, d)


def _timeit(fn, steps, warm):
    for _ in range(warm):
        fn()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    return (time.perf_counter() - t0) / steps


def cpu_reference(workload, batch, steps, warm):
    """The reference's own implementation of the workload on the host cores (fp32, all threads).  Returns
    (units/s, seconds/step, threads, kind, sample description).  kind "reference" = the unmodified scripts copied to oracle/_ref by
    oracle/build_ref.py drive the step through their own public API; "port" = the oracle restatement (when that copy is absent)."""
    import synth
    from test_oracle_golden import ma_synth_state
    torch.set_num_threads(os.cpu_count() or 1)
    threads = torch.get_num_threads()
    quiet = contextlib.redirect_stdout(io.StringIO())
    if workload == "ma_train":
        B = batch or PER_GPU_BATCH
        x, y = synth_batch(B, 1234)
        cad = _ref_module("causal_anomaly_detection")
        if cad is not None:
            # cad.train_model IS the reference's public training API (cad:609-790): AdamW(3e-4, wd 1e-5), clip 1.0, frozen stem, one epoch
            # over a list of `steps` batches, no validation batches.  Python loops (detector, tracker, per-clip GRU/VAE) included.
            cad.device = torch.device("cpu")
            torch.manual_seed(0)
            model = cad.CausalAnomalyDetector()
            model.load_state_dict(ma_synth_state(3, False), strict=True)

            def run(n):
                with quiet:
                    cad.train_model(model, [(x, y)] * n, [], num_epochs=1, lr=3e-4)
            if warm:
                run(warm)
            t0 = time.perf_counter()
            run(steps)
            dt = (time.perf_counter() - t0) / steps
            return B / dt, dt, threads, "reference", f"{B} clips/step x {steps} steps through causal_anomaly_detection.train_model (oracle/_ref, unmodified), fp32 CPU"
        from oracle import train as o_train
        P = ma_synth_state(3, False)
        opt = o_train.OracleAdam(o_train.ma_trainable(P), 3e-4, 1e-5, True, 1.0)
        eps, keep = ma_noise_for(B, 1234)
        dt = _timeit(lambda: o_train.ma_train_step(P, opt, x, y, eps, keep), steps, warm)
        return B / dt, dt, threads, "port", f"{B} clips/step x {steps} steps, oracle port of cad:637-690 (fwd + 4-term loss + bwd + clip + AdamW), fp32 CPU"
    if workload in ("mc_infer", "mc_long"):
        Ts = [16] if workload == "mc_infer" else [64, 128, 256]
        B = batch or 4
        xs = [synth.mc_clips(B, t, 64, 64, 1234) for t in Ts]
        mc3 = _ref_module("minicausal_vad_complete3")
        g = gold("mc.pt")
        P = synth.synth_fill(g["init_state"], seed=g["state_seed"])
        for k in P:
            if k.startswith("classifier") and k.endswith("weight"):
                P[k] = P[k] * 3.0
        if mc3 is not None:
            with quiet:
                model = mc3.SimpleVideoAnomalyDetector()
            model.load_state_dict(P, strict=True)
            model.eval()

            def fn():
                with torch.no_grad():
                    for x in xs:
                        model(x)
            kind = "reference"
        else:
            from oracle import mc as o_mc

            def fn():
                with torch.no_grad():
                    for x in xs:
                        o_mc.mc_forward(P, x)
            kind = "port"
        dt = _timeit(fn, steps, warm)
        frames = B * sum(Ts)
        return frames / dt, dt, threads, kind, f"{B} clips x T={Ts} per step x {steps} steps, SimpleVideoAnomalyDetector.forward eval ({kind}), fp32 CPU"
    if workload == "mb_train":
        B = batch or 32
        x = synth.mb_clips_bright(B, 8, 64, 64, 1234)
        y = torch.zeros(B)
        ck = gold("best_improved_model.pth")
        s2 = _ref_module("avenue_training_script2")
        if s2 is not None:
            with quiet:
                tr = s2.ImprovedMiniCausalVAD(device="cpu")
            tr.model.load_state_dict(ck["model_state_dict"], strict=True)
            tr.optimizer.load_state_dict(ck["optimizer_state_dict"])

            def run(n):
                with quiet:
                    tr.train_epoch_improved([(x, y)] * n)        # s2:207-263, the reference's epoch API over an in-memory loader
            if warm:
                run(warm)
            t0 = time.perf_counter()
            run(steps)
            dt = (time.perf_counter() - t0) / steps
            return B / dt, dt, threads, "reference", f"{B} clips/step x {steps} steps through ImprovedMiniCausalVAD.train_epoch_improved (oracle/_ref), fp32 CPU"
        from oracle import train as o_train
        P = {k: v.clone() for k, v in ck["model_state_dict"].items()}
        opt = o_train.OracleAdam(list(P.keys()), 5e-4, 1e-3, True, 0.5)
        kf, kg = synth.keep_mask((B, 16), 0.3, 1), synth.keep_mask((B, 128), 0.3, 2)
        pseudo = (torch.rand(B, generator=synth.gen(3)) > 0.95).float()
        dt = _timeit(lambda: o_train.mb_train_step(P, opt, x, pseudo, kf, kg), steps, warm)
        return B / dt, dt, threads, "port", f"{B} clips/step x {steps} steps, oracle port of s2:221-238, fp32 CPU"
    if workload == "me_windows":
        frames = torch.rand(1200, 3, 64, 64, generator=synth.gen(78))
        starts = list(range(0, 1200 - 8, 4))
        bbox = _ref_module("avenue_training_script_bbox")
        if bbox is None:
            raise RuntimeError("me_windows has no oracle port: the reference copy oracle/_ref is required for its CPU arm")
        torch.manual_seed(0)
        with quiet:
            m = bbox.CausalAnomalyDetector().eval()
        m.load_state_dict(synth.synth_fill(m.state_dict(), 555), strict=True)

        def fn():           # bbox:392-415: one batch-1 forward per stride-4 window
            with torch.no_grad():
                for st in starts:
                    m(frames[st:st + 8].permute(1, 0, 2, 3).unsqueeze(0))
        dt = _timeit(fn, steps, warm)
        return len(starts) / dt, dt, threads, "reference", f"{len(starts)} batch-1 windows per step x {steps} steps, bbox model forward loop (bbox:392-415), fp32 CPU"
    raise ValueError(workload)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    metric, unit, desc = WORKLOADS[args.workload]
    # bounded sample: the M-A step is ~10 s of CPU work per 32-clip batch, so at most 3 timed steps and 1 warm-up; what was RUN is reported
    cap_s, cap_w = {"ma_train": (3, 1), "me_windows": (3, 1), "mb_train": (10, 2)}.get(args.workload, (20, 3))
    steps, warm = max(1, min(args.steps, cap_s)), max(0, min(args.warmup, cap_w))
    rate, dt, cores, kind, sample = cpu_reference(args.workload, args.batch, steps, warm)
    line = {
        "impl": "reference", "metric": metric, "value": rate, "unit": unit, "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "requested": {"steps": args.steps, "warmup": args.warmup}, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "name": args.workload, "where": "host CPU, rank 0 only"},
        "cpu_baseline": {"value": rate, "unit": unit, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": rate, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ============================================================================================ M-A train step (headline)
def profile_graph(make_graph, path, title, reps=5, spans=()):
    """Per-ABI-call time inside a replayed step graph (external CUDA events around EVERY call of libcvad_b200.so), written as a markdown
    table: where the step's microseconds go, including what is not ours (torch fills / RNG / copies) as the unbracketed rest.
    ``make_graph()`` captures the step and returns a zero-argument callable that replays it."""
    from cvad_b200 import ops
    ops.TIMED.clear()
    ops.TIMED_NAMES.add("*")
    ops.TIMED_CAPTURE_ONLY[0] = True
    replay = make_graph()
    ops.TIMED_CAPTURE_ONLY[0] = False
    ops.TIMED_NAMES.clear()
    acc = {k: 0.0 for k in ops.TIMED}
    span_acc = [0.0] * len(spans)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    total = 0.0
    for i in range(reps + 1):
        e0.record()
        replay()
        e1.record()
        torch.cuda.synchronize()
        if i:
            total += e0.elapsed_time(e1) / reps
            for k, v in ops.TIMED.items():
                acc[k] += sum(s.elapsed_time(e) for s, e in v) / reps
            for j, (a, b, _) in enumerate(spans):       # from the END of the last call named a to the START of the first call named b
                if a in ops.TIMED and b in ops.TIMED:
                    span_acc[j] += ops.TIMED[a][-1][1].elapsed_time(ops.TIMED[b][0][0]) / reps
    lines = [f"# per-call time inside the replayed {title} (external CUDA events, mean of {reps} replays)\n",
             f"step (instrumented graph) {total * 1e3:.0f} us; sum of bracketed calls {sum(acc.values()) * 1e3:.0f} us "
             "(calls on the side streams overlap the main chain, so the sum may exceed the step)\n",
             "| ABI call | calls | us | share of step |", "|---|---:|---:|---:|"]
    for k, v in sorted(acc.items(), key=lambda kv: -kv[1]):
        lines.append(f"| `{k}` | {len(ops.TIMED[k])} | {v * 1e3:.1f} | {100 * v / total:.1f}% |")
    for (a, b, label), v in zip(spans, span_acc):
        lines.append(f"\n{label}: {v * 1e3:.0f} us (end of `{a}` -> start of `{b}` on the main stream)")
    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")
    ops.TIMED.clear()


def profile_calls(tr, x_dev, y_dev, path, reps=5):
    def make():
        gp = tr.graphed_train_step(x_dev, y_dev)
        return lambda: gp(x_dev, y_dev)
    profile_graph(make, path, "M-A train-step graph (batch 32)", reps,
                  spans=[("cvad_pad_avgpool_bf16_fwd", "cvad_pad_avgpool_bf16_bwd", "dense tail on the critical path (detector ... loss ... classifier backward)"),
                         ("cvad_stem_space_to_depth_u8", "cvad_flat_conv3x3_fwd_stats_bf16", "stem (both passes + max-pool)"),
                         ("cvad_pad_avgpool_bf16_bwd", "cvad_sumsq_f32", "backbone backward")])


def ma_self_check(dev, precision, frames):
    """The FIRST step of the benchmarked configuration against the unmodified reference: rank 0's batch is exactly the input of the golden
    case ``c2_sat_train`` (tests/golden/ma_c2.pt, tools/make_golden.py), so one training forward / 4-term loss with the reference's
    injected dropout masks and VAE noise must reproduce the reference's loss and per-clip scores (1e-3 bf16 / 5e-5 fp32)."""
    from test_oracle_golden import ma_synth_state
    from cvad_b200.ma import CausalAnomalyDetector, MATrainer
    from cvad_b200.noise import FixedNoise
    c = gold("ma_c2.pt")["cases"][0]
    m = CausalAnomalyDetector()
    m.load_state_dict(ma_synth_state(c["seed"], c["live"]), strict=True)
    tr = MATrainer(m, dev, precision=precision)
    tr.model.train()
    eps, keep = ma_noise_for(c["B"], c["xseed"])
    tr.model.noise = FixedNoise({"eps": eps, **keep})
    x, y = synth_batch(c["B"], c["xseed"], frames)
    assert torch.equal(y, c["labels"])
    comp, out = tr.forward_backward(x.to(dev), y.to(dev))
    torch.cuda.synchronize()
    loss, want = float(comp[0]), float(c["loss"])
    sc = out["anomaly_scores"].detach().cpu()
    e_l = abs(loss - want) / abs(want)
    e_s = float((sc - c["anomaly_scores"]).abs().max() / c["anomaly_scores"].abs().max())
    tol = 1e-3 if precision == "bf16" else 5e-5
    res = {"fixture": "tests/golden/ma_c2.pt:c2_sat_train (unmodified reference, fp32 CPU)", "loss": loss, "reference_loss": want,
           "loss_rel_err": e_l, "score_max_rel_err": e_s, "tolerance": tol, "ok": bool(e_l < tol and e_s < tol)}
    if not res["ok"]:
        raise RuntimeError(f"bench self-check failed: {res}")
    del tr, m
    torch.cuda.empty_cache()
    return res


def run_ma_train(args, rank, local, world, dev, dp):
    from test_oracle_golden import ma_synth_state
    from cvad_b200 import ops
    from cvad_b200.ma import CausalAnomalyDetector, MATrainer
    import torch.distributed as dist

    B = args.batch or PER_GPU_BATCH
    check = None
    if rank == 0 and not args.no_check and B == PER_GPU_BATCH:
        check = ma_self_check(dev, args.precision, args.frames)
        trace(f"self-check ok: loss {check['loss']:.6f} vs reference {check['reference_loss']:.6f}")
    # every rank starts from the same state (the stock init's saturated detector, SURVEY fact 6) and then draws its own noise and data
    model = CausalAnomalyDetector()
    model.load_state_dict(ma_synth_state(3, False), strict=True)
    tr = MATrainer(model, dev, precision=args.precision, dp=dp)
    if dp is not None:
        dp.broadcast_parameters(tr.optimizer.arena, model=tr.model)
        torch.cuda.synchronize()
        trace("state broadcast")
    torch.manual_seed(1234 + rank)
    tr.model.train()
    x_host, y_host = synth_batch(B, 1234 + rank, args.frames)
    x_pin, y_pin = x_host.pin_memory(), y_host.pin_memory()
    x_dev, y_dev = x_host.to(dev), y_host.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    gs = None
    if args.no_graph:
        def step(x, y):
            comp, out = tr.train_step(x, y)
            return comp, out["anomaly_scores"]
    else:
        # the whole step (zero_grad, forward, loss, backward, all-reduce, clip+AdamW) is one CUDA graph (two around the all-reduce for N > 1)
        trace("batch resident; capturing the step")
        gs = tr.graphed_train_step(x_dev, y_dev)
        trace("step captured")
        x_dev, y_dev = gs.static_inputs

        def step(x, y):
            return gs(x, y)

    for _ in range(args.warmup):
        step(x_dev, y_dev)
    barrier()
    trace("warm-up done")
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n0 = ops.LAUNCHES[0]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        last = step(x_dev, y_dev)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    trace(f"timed region done ({ms / args.steps:.3f} ms/step)")
    launches = ops.LAUNCHES[0] - n0
    if args.dump_outputs and rank == 0:        # before the end-to-end steps below train the model further
        dump_outputs(args.dump_outputs, {"loss_components": last[0], "anomaly_scores": last[1], "parameters": tr.optimizer.arena.p})

    # ---- end to end: pinned host batch -> H2D -> step -> D2H loss, through the public trainer API.  Every step's batch starts in pinned
    # host memory and its loss is read back to the host.  With the graphed trainer the H2D copy of step i+1 is issued before step i's
    # loss is read, so it overlaps step i's compute (all copies are inside the timed region: K+1 batches are copied for K timed steps).
    def e2e_step(first):
        if args.no_graph:
            return step(x_pin.to(dev, non_blocking=True), y_pin.to(dev, non_blocking=True))[0]
        if first:
            gs.prefetch(x_pin, y_pin)
        out = gs.run_prefetched()[0]
        gs.prefetch(x_pin, y_pin)
        return out

    for i in range(2):
        float(e2e_step(i == 0)[0])
    barrier()
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    loss_host = float("nan")
    for i in range(args.steps):
        c = e2e_step(False)
        loss_host = float(c[0])
    t1.record()
    barrier()
    ms_e2e = t0.elapsed_time(t1)
    trace(f"e2e region done ({ms_e2e / args.steps:.3f} ms/step)")
    sampler.stop_flag = True

    # ---- dominant kernel family, timed live with CUDA events around every call
    conv_names = {"cvad_flat_conv3x3_fwd_bf16", "cvad_flat_conv3x3_fwd_stats_bf16", "cvad_flat_conv3x3_dgrad_bf16",
                  "cvad_flat_conv3x3_wgrad_bf16", "cvad_flat_conv3x3_wgrad_staged_bf16"} if args.precision == "bf16" \
        else {"cvad_conv_fwd_f32", "cvad_conv_dgrad_f32", "cvad_conv_wgrad_f32"}
    probe_steps = 5
    ops.TIMED.clear()
    ops.TIMED_NAMES.update(conv_names)
    gp = None
    if args.no_graph:
        for _ in range(2):
            tr.train_step(x_dev, y_dev)
        torch.cuda.synchronize()
        ops.TIMED.clear()
        for _ in range(probe_steps):
            tr.train_step(x_dev, y_dev)
        torch.cuda.synchronize()
        conv_ms = {k: sum(s.elapsed_time(e) for s, e in v) / probe_steps for k, v in ops.TIMED.items()}
        how = f"CUDA events around each ABI call over {probe_steps} eager steps after the timed region"
    else:
        # a second capture of the same step with an (external) CUDA event pair around every convolution call: the events are
        # nodes of the graph, so each replay times the kernels exactly as they run inside the benchmarked step
        ops.TIMED_CAPTURE_ONLY[0] = True
        gp = tr.graphed_train_step(x_dev, y_dev)
        ops.TIMED_CAPTURE_ONLY[0] = False
        ops.TIMED_NAMES.clear()
        conv_ms = {k: 0.0 for k in ops.TIMED}
        for i in range(probe_steps + 1):
            gp(x_dev, y_dev)
            torch.cuda.synchronize()
            if i:                                   # the first replay warms the instrumented graph up
                for k, v in ops.TIMED.items():
                    conv_ms[k] += sum(s.elapsed_time(e) for s, e in v) / probe_steps
        how = f"external CUDA events around each ABI call inside the replayed step graph, mean of {probe_steps} replays after the timed region"
    ops.TIMED_NAMES.clear()
    conv_launches = sum(len(v) for v in ops.TIMED.values()) // (probe_steps if args.no_graph else 1)
    if args.profile_calls and not args.no_graph and rank == 0:
        profile_calls(tr, x_dev, y_dev, args.profile_calls)
    if world > 1:
        t = torch.tensor([ms, ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = t.tolist()
    trace("kernel probe done")
    ops.TIMED.clear()
    del gs, gp                       # the captured graphs go before the process group does
    torch.cuda.synchronize()
    if rank != 0:
        return None
    tf_peak, hbm_peak, src = peaks()
    traffic, traffic_src = conv_family_traffic() if args.precision == "bf16" else (None, None)
    ms_step = ms / args.steps
    conv_total_ms = sum(conv_ms.values())
    flops_step = CONV_TRAIN_MFLOP * 1e6 * B * T
    achieved = flops_step / (conv_total_ms / 1e3) / 1e12 if conv_total_ms > 0 else 0.0
    metric, unit, desc = WORKLOADS["ma_train"]
    in_bytes = x_pin.numel() * x_pin.element_size() + y_pin.numel() * 8
    line = {
        "metric": metric, "value": world * B / (ms_step / 1e3), "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": {"workload": desc, "name": "ma_train", "per_gpu_batch": B, "frames_per_clip": T, "frame": [H, W], "parallelism": f"dp{world}",
                   "l2": f"inputs ({in_bytes / 1e6:.0f} MB per step) and every layer's activations (99-375 MB) larger than the 126 MB L2",
                   "launch": "eager" if args.no_graph else "one CUDA graph per step",
                   "frames": "uint8 grayscale frames as the loader reads them (cad:89-96), Normalize(0.5,0.5) applied on the device "
                             "(bit-identical to the host-side fp32 path)" if args.frames == "u8" else "fp32 frames normalised on the host (cad:1177-1179)",
                   "e2e_path": "pinned host batch -> H2D (copy stream, overlapped with the previous step) -> graph -> D2H loss",
                   "initial_state": "synth_fill seed 3 (stock detector-bias init: saturated detector), identical on every rank",
                   "precision": ("bf16 operands, fp32 accumulate (tcgen05 kind::f16) in the eight 3x3 layers; stem: fp16 operands (the uint8 frames and "
                                 "their Normalize(0.5,0.5) images are exact in fp16), fp32 accumulate; dense tail fp32 (6144-wide projections 3xTF32)")
                   if args.precision == "bf16" else "fp32"},
        "e2e": {"value": world * B / (ms_e2e / args.steps / 1e3), "unit": unit, "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches,
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": tf_peak, "unit": "TFLOP/s", "frac": achieved / tf_peak, "traffic": traffic,
                     "traffic_source": traffic_src, "algorithmic_bytes_per_step": CONV_ALG_BYTES,
                     "kernel": "flatconv / flatwgrad TMA+tcgen05 3x3 convolutions (fwd incl. BatchNorm statistics + dgrad + wgrad incl. its fold pass, 8 layers)"
                     if args.precision == "bf16" else "conv_gemm_kernel fp32",
                     "peak_source": src, "launches_per_step": conv_launches, "ms_per_step": conv_total_ms,
                     "share_of_step": conv_total_ms / ms_step, "per_kernel_ms": conv_ms,
                     "algorithmic_gflop_per_step": flops_step / 1e9, "how": how},
        "clocks": sampler.summary(),
        "loss": loss_host,
        "self_check": check,
    }
    return line


# ============================================================================================ the small models (C1, C3, C4, C5)
def run_small(args, rank, local, world, dev, dp):
    """M-C / M-B / M-E workloads: each step is one CUDA-graph replay of the model's forward (or train step) on a per-GPU batch."""
    import synth
    import torch.distributed as dist
    from cvad_b200 import ops
    from cvad_b200.graphs import GraphedStep
    wl = args.workload
    metric, unit, desc = WORKLOADS[wl]
    check = None
    extra = {}
    seed = 1234 + rank

    if wl in ("mc_infer", "mc_long"):
        from cvad_b200.mc import SimpleVideoAnomalyDetector
        Ts = [16] if wl == "mc_infer" else [64, 128, 256]
        B = args.batch or 4
        g = gold("mc.pt")
        P = synth.synth_fill(g["init_state"], seed=g["state_seed"])
        for k in P:
            if k.startswith("classifier") and k.endswith("weight"):
                P[k] = P[k] * 3.0
        model = SimpleVideoAnomalyDetector()
        model.load_state_dict(P, strict=True)
        model = model.to(dev).eval()
        hosts = [synth.mc_clips(B, t, 64, 64, seed) for t in Ts]
        with torch.no_grad():
            graphs = [GraphedStep(lambda x: (model(x),), (h.to(dev),)) for h in hosts]
        units = B * sum(Ts)
        # algorithmic bytes: the fp32 input once (16.4 KB per frame) + the 73 KB of weights (SURVEY.md 8d)
        alg_bytes = sum(h.numel() * 4 for h in hosts) + 18337 * 4
        alg_flops = 12.39e6 * units
        if wl == "mc_infer" and rank == 0 and B == 4:
            want = next(c for c in g["eval"] if c["weights"] == "synth" and (c["B"], c["T"], c["seed"]) == (4, 16, 1234))["scores"]
            got = graphs[0](hosts[0].to(dev))[0].cpu()
            err = float((got - want).abs().max() / want.abs().max())
            check = {"fixture": "tests/golden/mc.pt (unmodified reference, fp32 CPU)", "score_max_rel_err": err, "tolerance": 1e-5, "ok": err < 1e-5}
            if not check["ok"]:
                raise RuntimeError(f"bench self-check failed: {check}")

        def step_dev():
            for gph, s in zip(graphs, [gg.static_inputs[0] for gg in graphs]):
                gph(s)
            return graphs[-1].outputs[0]

        def named_outputs(last):
            return {f"scores_T{t}": gph.outputs[0] for t, gph in zip(Ts, graphs)}

        def make_profiled():
            with torch.no_grad():
                gps = [GraphedStep(lambda x: (model(x),), (h.to(dev),)) for h in hosts]
            return lambda: [gp(gp.static_inputs[0]) for gp in gps]
        pins = [h.pin_memory() for h in hosts]

        def step_e2e():
            outs = [gph(p)[0] for gph, p in zip(graphs, pins)]
            return [o.cpu() for o in outs]            # D2H of every batch's scores
        h2d, d2h = sum(p.numel() * 4 for p in pins), 4 * B * len(Ts)
        extra["per_T"] = Ts
    elif wl == "mb_train":
        from cvad_b200.mb import ImprovedMiniCausalVAD
        B = args.batch or 32
        tr = ImprovedMiniCausalVAD(device=dev, verbose=False)
        ck = gold("best_improved_model.pth")
        tr.model.load_state_dict(ck["model_state_dict"], strict=True)
        tr.optimizer.load_state_dict(ck["optimizer_state_dict"])
        tr.model.train()
        if rank == 0:
            # first: one step of the golden trajectory (tests/golden/mb.pt: the reference's loss from the shipped checkpoint + AdamW state)
            from cvad_b200.noise import FixedNoise
            tg = gold("mb.pt")["trajectory"]
            sd = tg["seeds"][0]
            snap = [t.clone() for t in (tr.optimizer.arena.p, tr.optimizer.arena.m, tr.optimizer.arena.v, tr.optimizer.arena.state)]
            noise0 = tr.model.noise
            tr.model.noise = FixedNoise({"feat": synth.keep_mask((8, 16), 0.3, sd + 1), "graph": synth.keep_mask((8, 128), 0.3, sd + 2)})
            comp = tr.train_step(synth.mb_clips_bright(8, 8, 64, 64, sd).to(dev), torch.zeros(8, device=dev), (tg["steps"][0]["u"] > 0.95).float().to(dev))
            got, want = float(comp[0]), tg["losses"][0]
            for t, s in zip((tr.optimizer.arena.p, tr.optimizer.arena.m, tr.optimizer.arena.v, tr.optimizer.arena.state), snap):
                t.copy_(s)
            tr.model.noise = noise0
            err = abs(got - want) / abs(want)
            check = {"fixture": "tests/golden/mb.pt trajectory step 0 (unmodified reference, fp32 CPU)", "loss": got, "reference_loss": want,
                     "loss_rel_err": err, "tolerance": 5e-5, "ok": err < 5e-5}
            if not check["ok"]:
                raise RuntimeError(f"bench self-check failed: {check}")
        if dp is not None:          # attached only now: the self-check step above ran on rank 0 alone
            dp.attach(tr.optimizer)
            tr.dp = dp
            dp.broadcast_parameters(tr.optimizer.arena, model=tr.model)
        torch.manual_seed(seed)
        x_host, y_host = synth.mb_clips_bright(B, 8, 64, 64, seed), torch.zeros(B)
        gph = tr.graphed_train_step(x_host.to(dev), y_host.to(dev))
        units = B
        alg_bytes = x_host.numel() * 4 + 188849 * 28        # the input once + 28 B/parameter of optimizer traffic (SURVEY.md 8d)
        alg_flops = 191.8e6 * B

        def step_dev():
            return gph(*gph.static_inputs)[0]

        def named_outputs(last):
            return {"loss_components": last, "parameters": tr.optimizer.arena.p}

        def make_profiled():
            gp = tr.graphed_train_step(x_host.to(dev), y_host.to(dev))
            return lambda: gp(*gp.static_inputs)
        xp, yp = x_host.pin_memory(), y_host.pin_memory()

        def step_e2e():
            return gph(xp, yp)[0].cpu()
        h2d, d2h = xp.numel() * 4 + yp.numel() * 4, 32
    elif wl == "me_windows":
        from cvad_b200 import me
        torch.manual_seed(0)
        model = me.CausalAnomalyDetector()
        model.load_state_dict(synth.synth_fill(model.state_dict(), 555), strict=True)
        model = model.to(dev).eval()
        frames = torch.rand(1200, 3, 64, 64, generator=synth.gen(78 + rank))
        starts = list(range(0, 1200 - 8, 4))            # bbox:392 -> 298 windows
        units = len(starts)
        alg_bytes = frames.numel() * 4                  # every frame once (the windows overlap by 4 frames: gathering them costs no HBM re-read in principle)
        alg_flops = 0.0
        f_dev = frames.to(dev)
        f_pin = frames.pin_memory()

        def step_dev():
            return me.score_windows_device(model, f_dev)

        def named_outputs(last):
            return dict(zip(("scores", "adjacency", "features"), last))

        def step_e2e():
            return me.score_windows(model, f_pin, device=dev)[1]
        h2d, d2h = f_pin.numel() * 4, units * (4 + 256 * 4 + model.feature_dim * 4)
        if rank == 0:
            # the reference's way on the same GPU: one batch-1 call per window (bbox:392-415), bounded sample of 60 windows
            n = 60
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for st in starts[:n]:
                me.predict_anomaly_for_clip(model, f_pin[st:st + 8].permute(1, 0, 2, 3), device=dev)
            torch.cuda.synchronize()
            extra["batch1_loop_clips_per_s_same_gpu"] = n / (time.perf_counter() - t0)
    else:
        raise ValueError(wl)
    if wl == "me_windows":
        make_profiled = None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_dev()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n0 = ops.LAUNCHES[0]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        last = step_dev()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = ops.LAUNCHES[0] - n0
    if args.dump_outputs and rank == 0:        # before the end-to-end steps below (mb_train: they train the model further)
        dump_outputs(args.dump_outputs, named_outputs(last))
    for _ in range(2):
        step_e2e()
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.steps):
        res = step_e2e()
    t1.record()
    barrier()
    ms_e2e = t0.elapsed_time(t1)
    sampler.stop_flag = True
    if args.profile_calls and rank == 0 and make_profiled is not None:
        profile_graph(make_profiled, args.profile_calls, f"{wl} step graph")
    if world > 1:
        t = torch.tensor([ms, ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = t.tolist()
    torch.cuda.synchronize()
    if rank != 0:
        return None
    tf_peak, hbm_peak, src = peaks()
    ms_step = ms / args.steps
    gbs = alg_bytes / (ms_step / 1e3) / 1e9
    line = {
        "metric": metric, "value": world * units / (ms_step / 1e3), "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "name": wl, "per_gpu_units_per_step": units, "parallelism": f"dp{world}" if wl == "mb_train" else f"{world} independent clip shards",
                   "l2": "working set far below the 126 MB L2 and the step is launch/latency-bound: no flush between steps (stated, not hidden)",
                   "launch": "CUDA graph replay" if wl != "me_windows" else "eager (gather + batched forward)", **extra},
        "e2e": {"value": world * units / (ms_e2e / args.steps / 1e3), "unit": unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak, "traffic": None,
                     "kernel": "whole step (fp32 implicit-GEMM conv3d + BN/pool + dense tail); algorithmic bytes = the input once + weights"
                               " (SURVEY.md 8d): these models are launch/latency-bound at the reference's batch sizes",
                     "algorithmic_bytes_per_step": alg_bytes, "algorithmic_gflop_per_step": alg_flops / 1e9, "peak_source": src,
                     "how": "algorithmic bytes / CUDA-event time of the timed region"},
        "clocks": sampler.summary(),
        "self_check": check,
    }
    return line


def run_ours(args):
    # NCCL prints its version banner on stdout when NCCL_DEBUG=VERSION is set in the image; stdout carries exactly one JSON line
    if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", ""):
        os.environ["NCCL_DEBUG"] = "WARN"
    import torch.distributed as dist
    import cvad_b200  # noqa: F401
    from cvad_b200.parallel import DataParallel, init_from_env

    trace("imports done")
    # NCCL writes its version banner to the process's stdout when the first communicator is created (the image sets NCCL_DEBUG=VERSION for
    # child processes): stdout must carry exactly one JSON line, so file descriptor 1 points at stderr until that line is printed
    saved_stdout = os.dup(1)
    sys.stdout.flush()
    os.dup2(2, 1)
    rank, local, world = init_from_env()
    trace(f"process group up (world {world})")
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    dp = DataParallel() if world > 1 else None
    line = (run_ma_train if args.workload == "ma_train" else run_small)(args, rank, local, world, dev, dp)
    if rank == 0:
        if world == 1 and not args.no_cpu:
            steps, warm = (2, 1) if args.workload == "ma_train" else (10, 2)
            rate, dt, cores, kind, sample = cpu_reference(args.workload, args.batch, steps, warm)
            line["cpu_baseline"] = {"value": rate, "unit": line["unit"], "cores": cores, "kind": kind, "sample": sample}
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        # orderly teardown (the captured graphs are gone by now): every rank drains its GPU, meets at a barrier, then drops the group
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="ma_train", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (0 = the workload's BASELINE.json value)")
    ap.add_argument("--frames", default="u8", choices=["u8", "f32"], help="ma_train: what crosses PCIe -- the loader's uint8 frames or host-normalised fp32")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-check", action="store_true", help="skip the golden-fixture self-check of the first step")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of replaying one CUDA graph")
    ap.add_argument("--profile-calls", default="", help="write a per-ABI-call timing table of the replayed step graph to this file")
    ap.add_argument("--watchdog", type=int, default=420, help="seconds after which a stuck run dumps its stack and exits non-zero")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step returned to DIR/<name>.npy (float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    import faulthandler
    faulthandler.dump_traceback_later(args.watchdog, exit=True)     # a hang must never eat the GPU budget
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
    faulthandler.cancel_dump_traceback_later()
    sys.stdout.flush()
    sys.stderr.flush()


if __name__ == "__main__":
    main()
