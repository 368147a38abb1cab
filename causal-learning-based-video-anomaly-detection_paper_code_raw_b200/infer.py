"""Low-latency inference for the per-frame (2-D backbone) models M-A and M-A0.

``FrozenBackbone`` is the bf16 tensor-core backbone of tc.py specialised to eval mode.  An eval-mode BatchNorm is a constant per-channel
affine map, so it is folded into the convolution in front of it once, at snapshot time (w' = w*s, b' = (b - running_mean)*s + beta,
s = gamma / sqrt(running_var + eps)), and every 3x3 layer is ONE launch whose tcgen05 epilogue writes relu(conv + b') straight into the
layout the next layer reads.  Per call:

  x (n,1,H,W) uint8 / fp32 --stem: space-to-depth, conv + bn1 + ReLU + max-pool--> a0 --8 x flatconv relu--> a8 --avg-pool--> (n, 6144)

11 ABI calls (the training-shaped eval path of tc._BackboneBF16 takes 36: weight packs, BatchNorm prepares, a separate apply pass that
reads every convolution output back from HBM).  The numbers differ from that path in the last bits of bf16: the folded weights are
rounded as bf16(w*s) instead of bf16(w) followed by an fp32 affine map, and the pre-activation is not rounded to bf16 before the ReLU.

``MultiStreamScorer`` is ``ma0.StreamingWindowScorer`` for S streams at once with every push of a given size replayed as one CUDA graph:
each stream's position lives in a device-side cursor and each push carries a small descriptor (frames kept, start over) per stream, so
the same graph serves every push of that size whatever the streams' phases.  ``GraphedStreamingScorer`` is its one-stream case.
"""
from __future__ import annotations

import torch

from . import ops, tc
from .graphs import GraphedStep
from .ops import _call, _ptr, _st

BF16 = tc.BF16


class FrozenBackbone:
    """A snapshot of an eval-mode ``ma.ResNetBackbone`` (M-A's and M-A0's backbone) for inference: ``__call__(x)`` maps (n, 1, H, W)
    uint8 (raw frames) or fp32 (normalised) frames on the device to (n, 6144) fp32 features.

    Before every call the ``_version`` and ``data_ptr`` of each backbone parameter and buffer are compared with the snapshot: an in-place
    change (an optimizer step, ``load_state_dict``) is re-folded into the SAME buffers, so CUDA graphs that captured a call stay valid; a
    tensor replaced by a new one drops the snapshot and builds new buffers (``refresh`` then returns True)."""

    def __init__(self, backbone):
        if backbone.training:
            raise RuntimeError("FrozenBackbone needs backbone.eval(): it folds the BatchNorm running statistics into the convolutions")
        conv1 = backbone.conv1
        if conv1.out_channels != 32 or conv1.in_channels != 1 or conv1.kernel_size != (7, 7) or conv1.stride != (2, 2):
            raise RuntimeError("the tensor-core stem implements the reference's 7x7 stride-2 1->32 convolution (cad:115)")
        ops._cuda(conv1.weight)
        self.backbone = backbone
        self.layers = tc._layers(backbone)
        self.strides = [conv.stride[0] for conv, _ in self.layers]
        if self.strides[0] == 2:
            raise RuntimeError("the first 3x3 convolution after the stem is stride 1 in the reference (cad:150)")
        self._acts = {}           # (n, H, W) -> persistent activation buffers, zeroed once
        self._snapshot()

    def _tensors(self):
        return list(self.backbone.parameters()) + list(self.backbone.buffers())

    def _state(self):
        return [(t._version, t.data_ptr()) for t in self._tensors()]

    def _snapshot(self):
        dev = self.backbone.conv1.weight.device
        f32 = dict(device=dev, dtype=torch.float32)
        self.mean1 = torch.empty(self.backbone.conv1.out_channels, **f32)
        self.invstd1 = torch.empty_like(self.mean1)
        self.folded = []          # per layer: (w' fp32 OIHW, b' fp32, w' packed bf16 for the forward)
        for conv, _ in self.layers:
            cout, cin = conv.out_channels, conv.in_channels
            if conv.kernel_size != (3, 3) or conv.padding != (1, 1):
                raise RuntimeError("the flat tensor-core convolution implements the reference's 3x3 / padding 1 layers (cad:128-139)")
            self.folded.append((torch.empty((cout, cin, 3, 3), **f32), torch.empty(cout, **f32),
                                torch.empty((9 * cout, cin), device=dev, dtype=BF16)))
        self._fold()

    def _fold(self):
        """Eval prepare of bn1, then fold + pack of every 3x3 layer, into the snapshot's buffers."""
        bb, st = self.backbone, _st()
        bn1 = bb.bn1
        _call("cvad_bn_eval_prepare_f32", bb.conv1.out_channels, float(bn1.eps), _ptr(bn1.running_mean), _ptr(bn1.running_var), _ptr(self.mean1),
              _ptr(self.invstd1), st)
        for (conv, bn), (wf, bf, wp), stride in zip(self.layers, self.folded, self.strides):
            w = ops._f32c(conv.weight.detach())
            cout, cin = conv.out_channels, conv.in_channels
            _call("cvad_bn_fold_conv_f32", _ptr(w), _ptr(conv.bias), _ptr(bn.weight), _ptr(bn.bias), _ptr(bn.running_mean), _ptr(bn.running_var),
                  float(bn.eps), cout, 9 * cin, _ptr(wf), _ptr(bf), st)
            _call("cvad_flat_pack_w3x3_bf16", _ptr(wf), cout, cin, stride, _ptr(wp), None, st)
        self._seen = self._state()

    @torch.no_grad()
    def refresh(self) -> bool:
        """Bring the snapshot up to date with the backbone.  Returns True when the buffers were replaced (a backbone tensor was)."""
        state = self._state()
        if state == self._seen:
            return False
        if len(state) != len(self._seen) or any(a[1] != b[1] for a, b in zip(state, self._seen)):
            self._snapshot()
            return True
        self._fold()
        return False

    def _buffers(self, n, H, W, dev):
        key = (n, H, W)
        bufs = self._acts.get(key)
        if bufs is None:
            # zeroed once: the phase-plane epilogue never writes the plane positions that have no source pixel
            h, w = tc.out_hw(*tc.out_hw(H, W, 2), 2)
            bufs = [torch.zeros(tc.act_shape(n, h, w, self.backbone.conv1.out_channels, False), device=dev, dtype=BF16)]
            for i, (conv, _) in enumerate(self.layers):
                h, w = tc.out_hw(h, w, self.strides[i])
                phase_out = i + 1 < len(self.layers) and self.strides[i + 1] == 2
                bufs.append(torch.zeros(tc.act_shape(n, h, w, conv.out_channels, phase_out), device=dev, dtype=BF16))
            self._acts[key] = bufs
        return bufs

    @torch.no_grad()
    def __call__(self, x):
        ops._cuda(x)
        if self.backbone.training:
            raise RuntimeError("FrozenBackbone needs backbone.eval(): it folds the BatchNorm running statistics into the convolutions")
        if x.dim() != 4 or x.shape[1] != 1 or x.dtype not in (torch.uint8, torch.float32):
            raise ValueError("expected (n, 1, H, W) uint8 or float32 frames")
        self.refresh()
        x = x.contiguous()
        n, _, H, W = x.shape
        st = _st()
        acts = self._buffers(n, H, W, x.device)
        tc.stem_forward(self.backbone, x, acts[0], self.mean1, self.invstd1)
        h, w = tc.out_hw(*tc.out_hw(H, W, 2), 2)
        cin = self.backbone.conv1.out_channels
        for i, ((conv, _), (_, bf, wp)) in enumerate(zip(self.layers, self.folded)):
            phase_out = i + 1 < len(self.layers) and self.strides[i + 1] == 2
            _call("cvad_flat_conv3x3_fwd_relu_bf16", _ptr(acts[i]), _ptr(wp), _ptr(bf), _ptr(acts[i + 1]), n, h, w, cin, conv.out_channels,
                  self.strides[i], int(phase_out), st)
            h, w = tc.out_hw(h, w, self.strides[i])
            cin = conv.out_channels
        feats = torch.empty((n, cin, 4, 6), device=x.device, dtype=torch.float32)
        _call("cvad_pad_avgpool_bf16_fwd", _ptr(acts[-1]), n, h, w, cin, 4, 6, _ptr(feats), st)
        return feats.reshape(n, -1)


def window_count(n_frames, next_window, count, reset, clip_len, stride):
    """The window rule of one stream for one push (the host's copy of ``stream_push`` in ma0_tail.cu): a stream that has seen
    ``n_frames`` frames and scored windows [0, ``next_window``) receives ``count`` frames (after starting over at frame 0 when ``reset``).
    Window w covers frames w*stride + [0, clip_len).  Returns (frames seen after the push, windows the push completes)."""
    base, nxt = (0, 0) if reset else (n_frames, next_window)
    frames = base + count
    return frames, ((frames - clip_len) // stride + 1 - nxt if frames >= clip_len else 0)


class MultiStreamScorer:
    """Sliding-window scoring of S frame streams (cameras, or the videos of a test set, bbox:392-430) with one CUDA graph replay per push
    for all of them.  Each stream gets exactly the windows and scores it would get from its own ``GraphedStreamingScorer``.

    ``push(frames, counts)`` takes n new frames per stream, of which stream k keeps the first ``counts[k]``, and runs: copy into static
    inputs -> ``FrozenBackbone`` over all S*n frames -> write each stream's kept feature rows into its ring at its device cursor -> gather
    the windows each stream completed (m slots per stream, m = the most any stream completed; unused slots are zeros) -> ``model.tail``
    over the S*m slots -> advance the cursors.  The counts and the streams to start over (``reset``) travel in a small per-push descriptor
    that is a static input of the graph, so raggedness does not capture again: the graph key is (n, m, H, W, dtype), and since a stream
    completes at most ceil(n / stride) windows in a push, a scorer holds at most ceil(n / stride) + 1 graphs per push size.  The host
    mirrors every cursor (``n_frames``, ``next_window``) with ``window_count``, so it knows m and each stream's part of the output
    without a device sync.  Graphs share one memory pool, read the model's live tensors (in-place weight updates need nothing) and are
    dropped when a model tensor is replaced by a new one."""

    def __init__(self, model, streams, clip_len=16, stride=4, capacity=64):
        if model.training:
            raise RuntimeError(f"{type(self).__name__} needs model.eval(): train-mode BatchNorm couples the frames of a batch")
        if capacity < clip_len + stride:
            raise ValueError("ring capacity must hold at least one window plus one stride of new frames")
        if streams < 1:
            raise ValueError("a scorer needs at least one stream")
        self.model, self.streams = model, int(streams)
        self.clip_len, self.stride, self.capacity = int(clip_len), int(stride), int(capacity)
        self.frozen = None
        self.rings = None           # (S, capacity, F) fp32 on the model's device
        self.cursors = None         # (S, 2) int64 {frames pushed, next window} per stream on the device: what the graphs read
        self._n_frames = [0] * self.streams          # host mirrors of the cursors: they decide m, the output slices and the graph key
        self._next_window = [0] * self.streams
        self._reset = [False] * self.streams         # streams the next push starts over
        self.graphs = {}            # (n, m, H, W, dtype) -> GraphedStep
        self.pool = None
        self._ptrs = None

    @property
    def n_frames(self):
        """Frames each stream has pushed since its last start."""
        return list(self._n_frames)

    @property
    def next_window(self):
        """Index of each stream's next window."""
        return list(self._next_window)

    def reset(self, k):
        """Start stream k over (a new video on that camera): the next push writes its frames from frame 0 and window 0 on."""
        if not 0 <= k < self.streams:
            raise IndexError(f"stream {k} out of range for {self.streams} streams")
        self._n_frames[k] = self._next_window[k] = 0
        self._reset[k] = True

    def _model_ptrs(self):
        return [t.data_ptr() for t in list(self.model.parameters()) + list(self.model.buffers())]

    def _step(self, n, m):
        model, S, T, F = self.model, self.streams, self.clip_len, self.rings.shape[2]

        def step(x, push):
            feats = self.frozen(x.reshape(S * n, *x.shape[2:]))
            st = _st()
            _call("cvad_streams_ring_write_f32", _ptr(feats), S, n, F, _ptr(self.rings), self.capacity, T, self.stride, _ptr(self.cursors),
                  _ptr(push), st)
            if m > 0:
                clips = torch.empty((S * m, T, F), device=feats.device, dtype=torch.float32)
                _call("cvad_streams_window_features_f32", _ptr(self.rings), S, self.capacity, self.stride, T, F, m, _ptr(self.cursors),
                      _ptr(push), _ptr(clips), st)
                scores = model.tail(clips)["anomaly_scores"]
            else:
                scores = torch.empty(0, device=feats.device)
            _call("cvad_streams_cursor_advance", _ptr(self.cursors), S, T, self.stride, _ptr(push), st)
            return scores
        return step

    @torch.no_grad()
    def push(self, frames, counts=None):
        """frames (S,n,1,H,W) float32 (normalised) or uint8 (the loader's raw frames) on the model's device; counts: S ints in [0, n], the
        frames each stream keeps (default n; the rows beyond a count are computed and discarded, so they must hold finite frames).
        Returns one (window scores, first window index) pair per stream; a stream's scores may be empty."""
        if frames.dim() != 5:
            raise ValueError("expected (S, n, 1, H, W) frames")
        S, n = self.streams, frames.shape[1]
        if frames.shape[0] != S:
            raise ValueError(f"expected frames of {S} streams, got {frames.shape[0]}")
        counts = [n] * S if counts is None else [int(c) for c in counts]
        if len(counts) != S or not all(0 <= c <= n for c in counts):
            raise ValueError(f"counts must be {S} ints in [0, {n}]")
        if max(counts) > self.capacity - self.clip_len:
            raise ValueError("more new frames than the ring can take while it still holds an open window")
        ops._cuda(frames)
        if self.model.training:
            raise RuntimeError(f"{type(self).__name__} needs model.eval(): train-mode BatchNorm couples the frames of a batch")
        bb = self.model.backbone
        if self.frozen is None or self.frozen.backbone is not bb:
            self.frozen = FrozenBackbone(bb)
            self.graphs.clear()
        replaced = self.frozen.refresh()
        ptrs = self._model_ptrs()
        if replaced or ptrs != self._ptrs:
            self.graphs.clear()
            self._ptrs = ptrs
        dev = frames.device
        if self.rings is None:
            F = bb.layer4[3].out_channels * 4 * 6
            self.rings = torch.zeros((S, self.capacity, F), device=dev, dtype=torch.float32)
            self.cursors = torch.zeros((S, 2), device=dev, dtype=torch.int64)
            self.pool = torch.cuda.graph_pool_handle()
        w0 = list(self._next_window)
        if not any(counts):         # nothing to write; pending resets reach the device with the next push
            empty = torch.empty(0, device=dev)
            return [(empty, w) for w in w0]
        wins = [window_count(self._n_frames[k], self._next_window[k], counts[k], self._reset[k], self.clip_len, self.stride) for k in range(S)]
        m = max(nw for _, nw in wins)
        push = torch.tensor([[c, int(r)] for c, r in zip(counts, self._reset)], dtype=torch.int64)
        key = (n, m, frames.shape[3], frames.shape[4], frames.dtype)
        g = self.graphs.get(key)
        if g is None:
            self.frozen._buffers(S * n, frames.shape[3], frames.shape[4], dev)      # allocated and zeroed outside the capture
            # warm-up runs the step for real: the rings and the cursors are restored after it, so capturing does not advance the streams
            g = self.graphs[key] = GraphedStep(self._step(n, m), (frames, push), mutated=(self.rings, self.cursors), pool=self.pool)
        (scores,) = g(frames, push)
        for k, (fr, nw) in enumerate(wins):
            self._n_frames[k] = fr
            self._next_window[k] += nw
        self._reset = [False] * S
        out = scores.clone()
        return [(out[k * m:k * m + nw], w0[k]) for k, (_, nw) in enumerate(wins)]


class GraphedStreamingScorer(MultiStreamScorer):
    """Sliding-window scoring of one frame stream, as ``ma0.StreamingWindowScorer`` (same constructor, ``push`` contract and errors), with
    each push replayed as one CUDA graph: ``MultiStreamScorer`` with one stream.  Each distinct (n, n_win, H, W, dtype) is captured once.
    Use it for a fixed chunk size and a model that is frozen or updated in place; a stream of ever-changing chunk sizes pays one capture
    per new size."""

    def __init__(self, model, clip_len=16, stride=4, capacity=256):
        super().__init__(model, 1, clip_len, stride, capacity)

    ring = property(lambda self: None if self.rings is None else self.rings[0], doc="(capacity, F) fp32 ring on the model's device")
    cursor = property(lambda self: None if self.cursors is None else self.cursors[0], doc="int64 {frames pushed, next window} on the device")
    n_frames = property(lambda self: self._n_frames[0], doc="frames pushed so far")
    next_window = property(lambda self: self._next_window[0], doc="index of the next window")

    def push(self, frames):
        """frames (n,1,H,W) float32 (normalised) or uint8 (the loader's raw frames) on the model's device -> (window scores, first window index)."""
        if frames.dim() != 4:
            raise ValueError("expected (n, 1, H, W) frames")
        [(scores, w0)] = super().push(frames.unsqueeze(0))
        return scores, w0
