"""CUDA-graph capture of a whole train / inference step (forward, fused loss, backward, all-reduce, fused clip+Adam).

A step of the hot path is 250-300 kernel launches of a few microseconds each; issued one by one from Python the host
is slower than the device (~17 ms of launch work for a ~10 ms step).  Every kernel of libcvad_b200.so launches on the
caller's stream, allocates nothing and never synchronises, and all step bookkeeping (NaN flags, skip logic, Adam step
counts) lives on the device, so the whole step can be captured once and replayed with one launch.

Capturing needs a few warm-up executions on a side stream (lazy one-time initialisation: function attributes, driver
entry points, torch's allocator).  Those executions are real steps, so every tensor a step mutates -- parameters, Adam
moments and counters, BatchNorm running statistics -- is snapshotted before and restored after them: building the graph
does not advance training.
"""
from __future__ import annotations

import torch

from . import ops


class GraphedStep:
    """``step_fn(*static_inputs) -> tuple of tensors`` captured into one CUDA graph.

    ``__call__(*inputs)`` copies the inputs into the static buffers (an H2D copy when they live in pinned host memory),
    replays the graph and returns the static output tensors (valid until the next replay)."""

    def __init__(self, step_fn, example_inputs, mutated=(), warmup: int = 3, pre_replay=None, between=None, tail_fn=None, stages=None,
                 pool=None):
        """``between`` / ``tail_fn`` split the step in two graphs around an eagerly issued call: graph(step_fn) ->
        between() -> graph(tail_fn).  The data-parallel trainer uses it to keep the NCCL gradient all-reduce OUT of the
        captured graphs (``between``) while forward/backward and the fused optimizer are each one graph launch.

        ``stages``: the general form, a list ``[(eager_fn or None, graph_fn), ...]`` run after ``step_fn``'s graph: for every entry
        the eager callable is issued on the current stream (e.g. an asynchronous collective), then the graph of ``graph_fn()`` is
        replayed.  All graphs share one memory pool, so later stages may use tensors that earlier stages produced.

        ``pool``: a memory pool handle (``torch.cuda.graph_pool_handle()``) to capture into, shared with other steps that are never
        replayed concurrently with this one (default: a private pool)."""
        self.pre_replay = pre_replay
        if stages is None:
            stages = [(between, tail_fn)] if (between is not None or tail_fn is not None) else []
        self.stages = [(e, f, None) for e, f in stages]
        self.static_inputs = [torch.empty_like(t, device=t.device if t.is_cuda else torch.cuda.current_device()) for t in example_inputs]
        for s, t in zip(self.static_inputs, example_inputs):
            s.copy_(t)
        mutated = [t for t in mutated if t is not None]
        snap = [t.detach().clone() for t in mutated]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                step_fn(*self.static_inputs)
                for eager, fn, _g in self.stages:
                    if eager is not None:
                        eager()
                    if fn is not None:
                        fn()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        with torch.no_grad():
            for t, s in zip(mutated, snap):
                t.copy_(s)
        del snap
        self.graph = torch.cuda.CUDAGraph()
        n0 = ops.LAUNCHES[0]
        with torch.cuda.graph(self.graph, pool=pool):
            out = step_fn(*self.static_inputs)
        pool = self.graph.pool()
        captured = []
        for eager, fn, _g in self.stages:
            g = None
            if fn is not None:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, pool=pool):
                    fn()
            captured.append((eager, fn, g))
        self.stages = captured
        self.launches = ops.LAUNCHES[0] - n0          # cvad ABI calls inside one replay
        self.outputs = out if isinstance(out, tuple) else (out,)

    def _replay(self):
        if self.pre_replay is not None:
            self.pre_replay()
        self.graph.replay()
        for eager, _fn, g in self.stages:
            if eager is not None:
                eager()
            if g is not None:
                g.replay()
        ops.LAUNCHES[0] += self.launches

    # ---- input prefetch: the H2D copy of batch i+1 runs on a copy stream while the graph of batch i executes
    def _init_prefetch(self):
        self.staging = [torch.empty_like(s) for s in self.static_inputs]
        self.copy_stream = torch.cuda.Stream()
        self.ev_ready, self.ev_free = torch.cuda.Event(), torch.cuda.Event()
        self.ev_free.record(torch.cuda.current_stream())

    def prefetch(self, *inputs):
        """Start copying the NEXT step's inputs (pinned host or device tensors) into a staging buffer, asynchronously."""
        if not hasattr(self, "staging"):
            self._init_prefetch()
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.ev_free)           # the previous step has consumed the staging buffer
            for st, t in zip(self.staging, inputs):
                st.copy_(t, non_blocking=True)
            self.ev_ready.record(self.copy_stream)

    def run_prefetched(self):
        """Run one step on the inputs handed to the last ``prefetch`` call."""
        cur = torch.cuda.current_stream()
        cur.wait_event(self.ev_ready)
        for s, st in zip(self.static_inputs, self.staging):
            s.copy_(st, non_blocking=True)                      # device-to-device, ~55 us for the 177 MB batch
        self.ev_free.record(cur)
        self._replay()
        return self.outputs

    def __call__(self, *inputs):
        for s, t in zip(self.static_inputs, inputs):
            if t is not s:
                s.copy_(t, non_blocking=True)
        self._replay()
        return self.outputs


def graphed_optimizer_step(opt, fwd_bwd, example_inputs, mutated, late_backward=None):
    """Capture ``fwd_bwd(*inputs) -> tuple`` (zero_grad + forward + loss + backward) followed by ``opt``'s fused step.

    Single GPU: one graph.  Data parallel (the optimizer carries a gradient all-reduce hook): the collective stays between graphs,
    because NCCL captured inside a graph stalled an 8-rank run (DESIGN.md section 4):
        graph(fwd_bwd) -> eager all-reduce -> graph(fused clip + Adam).
    ``late_backward``: an optional second part of the backward (M-A: the backbone's) whose gradients live in the arena range the hook
    calls "late".  Then the gradients ``fwd_bwd`` produced are reduced asynchronously WHILE the late backward runs:
        graph(fwd_bwd) -> start all-reduce(early range) -> graph(late_backward) -> all-reduce(late range), wait -> graph(clip + Adam)."""
    import os

    opt.sync_lr_to_device()
    hook = opt.pre_step_hook
    if hook is not None and os.environ.get("CVAD_NCCL_IN_GRAPH", "0") != "1":
        overlap = getattr(hook, "__self__", None)
        if late_backward is not None and overlap is not None and hasattr(overlap, "start_early") and os.environ.get("CVAD_ALLREDUCE_OVERLAP", "1") != "0":
            return GraphedStep(fwd_bwd, example_inputs, mutated, pre_replay=opt.sync_lr_to_device,
                               stages=[(lambda: overlap.start_early(opt.arena), late_backward),
                                       (lambda: overlap.finish_late(opt.arena), opt.step_local)])
        if late_backward is not None:
            def both(*inputs):
                out = fwd_bwd(*inputs)
                late_backward()
                return out
            return GraphedStep(both, example_inputs, mutated, pre_replay=opt.sync_lr_to_device,
                               between=lambda: hook(opt.arena), tail_fn=opt.step_local)
        return GraphedStep(fwd_bwd, example_inputs, mutated, pre_replay=opt.sync_lr_to_device,
                           between=lambda: hook(opt.arena), tail_fn=opt.step_local)

    def step(*inputs):
        out = fwd_bwd(*inputs)
        if late_backward is not None:
            late_backward()
        opt.step()
        return out
    return GraphedStep(step, example_inputs, mutated, pre_replay=opt.sync_lr_to_device)
