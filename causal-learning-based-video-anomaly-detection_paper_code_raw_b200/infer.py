"""Low-latency inference: the per-frame (2-D backbone) models M-A and M-A0, and many camera streams for the 3-D clip models and M-D.

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

``MultiStreamClipScorer`` is the same service for M-B, M-C and M-E from raw camera frames: the rings hold cv2-resized frames instead of
features, and every completed window is gathered from them and scored by the model's batched forward.

``MultiStreamAutoEncoderScorer`` is the same service for M-D: its eval-mode encoder is per frame, so each frame is encoded once into a ring
of LSTM input projections, and each completed window runs only the recurrence, the decoder and its score kernel.  The three multi-stream
scorers share their host-side bookkeeping (``_StreamBookkeeping``) and the device window rule (``stream_push``, mirrored by
``window_count``).
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


class _StreamBookkeeping:
    """The host side of S streams scored through device rings, shared by ``MultiStreamScorer`` (rings of backbone features) and
    ``MultiStreamClipScorer`` (rings of frames): constructor checks, push validation, the host mirrors of the device cursors
    (``window_count``), resets, the per-push descriptor, graph keys and capture, dropping the graphs when a model tensor is replaced, and
    the per-stream split of the outputs.  A subclass supplies its ring (``_new_ring``), the graph of one push (``_capture``), the outputs of
    a push that keeps no frame (``_empty``) and, optionally, its own check for replaced tensors (``_refresh``)."""

    def __init__(self, model, streams, clip_len, stride, capacity):
        if model.training:
            raise RuntimeError(f"{type(self).__name__} needs model.eval(): train-mode BatchNorm couples the frames of a batch")
        if capacity < clip_len + stride:
            raise ValueError("ring capacity must hold at least one window plus one stride of new frames")
        if streams < 1:
            raise ValueError("a scorer needs at least one stream")
        self.model, self.streams = model, int(streams)
        self.clip_len, self.stride, self.capacity = int(clip_len), int(stride), int(capacity)
        self.rings = None           # (S, capacity, ...) on the model's device
        self.cursors = None         # (S, 2) int64 {frames pushed, next window} per stream on the device: what the graphs read
        self._n_frames = [0] * self.streams          # host mirrors of the cursors: they decide m, the output slices and the graph key
        self._next_window = [0] * self.streams
        self._reset = [False] * self.streams         # streams the next push starts over
        self.graphs = {}            # (n, m, ...frame key) -> GraphedStep
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

    def _refresh(self):
        """Bring derived model state up to date; True when the graphs read tensors that no longer exist."""
        return False

    def _push(self, frames, counts, frame_key):
        """frames (S, n, ...) on the device -> per stream (tuple of its rows of every output, first window index)."""
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
        replaced = self._refresh()
        ptrs = self._model_ptrs()
        if replaced or ptrs != self._ptrs:
            self.graphs.clear()
            self._ptrs = ptrs
        dev = frames.device
        if self.rings is None:
            self.rings = self._new_ring(dev)
            self.cursors = torch.zeros((S, 2), device=dev, dtype=torch.int64)
            self.pool = torch.cuda.graph_pool_handle()
        w0 = list(self._next_window)
        if not any(counts):         # nothing to write; pending resets reach the device with the next push
            return [(self._empty(dev), w) for w in w0]
        wins = [window_count(self._n_frames[k], self._next_window[k], counts[k], self._reset[k], self.clip_len, self.stride) for k in range(S)]
        m = max(nw for _, nw in wins)
        push = torch.tensor([[c, int(r)] for c, r in zip(counts, self._reset)], dtype=torch.int64)
        key = (n, m) + frame_key
        g = self.graphs.get(key)
        if g is None:
            g = self.graphs[key] = self._capture(n, m, frames, push)
        outs = [o.clone() for o in g(frames, push)]
        for k, (fr, nw) in enumerate(wins):
            self._n_frames[k] = fr
            self._next_window[k] += nw
        self._reset = [False] * S
        return [(tuple(o[k * m:k * m + nw] for o in outs), w0[k]) for k, (_, nw) in enumerate(wins)]


class MultiStreamScorer(_StreamBookkeeping):
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
        super().__init__(model, streams, clip_len, stride, capacity)
        self.frozen = None

    def _refresh(self):
        bb = self.model.backbone
        new = self.frozen is None or self.frozen.backbone is not bb
        if new:
            self.frozen = FrozenBackbone(bb)
        return self.frozen.refresh() or new

    def _new_ring(self, dev):
        F = self.model.backbone.layer4[3].out_channels * 4 * 6
        return torch.zeros((self.streams, self.capacity, F), device=dev, dtype=torch.float32)

    def _empty(self, dev):
        return (torch.empty(0, device=dev),)

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

    def _capture(self, n, m, frames, push):
        self.frozen._buffers(self.streams * n, frames.shape[3], frames.shape[4], frames.device)      # allocated and zeroed outside the capture
        # warm-up runs the step for real: the rings and the cursors are restored after it, so capturing does not advance the streams
        return GraphedStep(self._step(n, m), (frames, push), mutated=(self.rings, self.cursors), pool=self.pool)

    @torch.no_grad()
    def push(self, frames, counts=None):
        """frames (S,n,1,H,W) float32 (normalised) or uint8 (the loader's raw frames) on the model's device; counts: S ints in [0, n], the
        frames each stream keeps (default n; the rows beyond a count are computed and discarded, so they must hold finite frames).
        Returns one (window scores, first window index) pair per stream; a stream's scores may be empty."""
        if frames.dim() != 5:
            raise ValueError("expected (S, n, 1, H, W) frames")
        return [(scores, w0) for (scores,), w0 in self._push(frames, counts, (frames.shape[3], frames.shape[4], frames.dtype))]


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


class MultiStreamClipScorer(_StreamBookkeeping):
    """Sliding-window scoring of S camera streams for the 3-D clip models -- M-B (``mb.CausalAnomalyDetector``, the model
    best_improved_model.pth loads into), M-E (``me.CausalAnomalyDetector``, bbox:392-430's window service) and M-C
    (``mc.SimpleVideoAnomalyDetector``) -- from raw uint8 frames, with one CUDA graph replay per push for all streams.

    Their temporal zero padding makes every window's activations depend on where the window starts (DESIGN.md section 5), so the rings hold
    resized FRAMES, and each completed window is gathered from its ring and scored by the model's own batched forward: the scores are
    those of ``model(clips)`` on the clips the reference builds per window.  ``push(frames, counts)`` runs: copy into static inputs ->
    resize each stream's kept frames into its ring at its device cursor (``cvad_streams_frame_write_u8``: cv2.resize INTER_LINEAR, bit
    for bit) -> gather the windows each stream completed into m fp32 clip slots per stream, unused slots zeros (``cvad_streams_clips_f32``)
    -> ``model`` over the S*m slots -> advance the cursors.  M-B and M-E take C = 3 frames in BGR order, as cv2 and video decoders deliver
    them, and see RGB clips in [0, 1] (the Avenue / bbox loader rule, bbox:397-411); M-C takes C = 1 grayscale frames, scaled by 1/255.
    M-C's reference loader resizes with PIL (mc3:104-216), not cv2: push M-C frames already at the model's size, where the ring write is
    a copy.

    Window w of a stream covers its frames w*stride + [0, clip_len) and is scored as soon as they have arrived, the rule of
    ``MultiStreamScorer`` (``window_count``).  bbox's loop over a finished video, ``range(0, F - window, stride)``, stops one window earlier
    when (F - clip_len) % stride == 0: such a video gets one window more here, its last one.

    Counts, ``reset``, ``n_frames``, ``next_window`` and the errors are those of ``MultiStreamScorer``.  The graph key is
    (n, m, H, W, C): at most ceil(n / stride) + 1 graphs per push size and camera frame size.  Graphs share one memory pool and read the
    model's live tensors, so an in-place weight or BatchNorm-statistic update needs no capture (M-C's eval BatchNorm fold runs inside the
    graph); a replaced tensor drops them."""

    def __init__(self, model, streams, clip_len=8, stride=4, capacity=32, size=(64, 64)):
        from . import mb, mc, me
        if isinstance(model, (mb.CausalAnomalyDetector, me.CausalAnomalyDetector)):
            self.channels, self.reverse_channels = 3, 1
            v = 16 if isinstance(model, me.CausalAnomalyDetector) else model.causal_discovery.num_variables
            feat = model.feature_dim if isinstance(model, me.CausalAnomalyDetector) else model.feature_extractor.fc.out_features
            self._out_shapes = ((), (v, v), (feat,))
        elif isinstance(model, mc.SimpleVideoAnomalyDetector):
            self.channels, self.reverse_channels = 1, 0
            self._out_shapes = ((),)
        else:
            raise TypeError(f"MultiStreamClipScorer scores mb.CausalAnomalyDetector, me.CausalAnomalyDetector or mc.SimpleVideoAnomalyDetector, "
                            f"not {type(model).__name__}")
        super().__init__(model, streams, clip_len, stride, capacity)
        self.size = (int(size[0]), int(size[1]))          # (width, height), as cv2.resize takes it

    def _new_ring(self, dev):
        w, h = self.size
        return torch.zeros((self.streams, self.capacity, h, w, self.channels), device=dev, dtype=torch.uint8)

    def _empty(self, dev):
        return tuple(torch.empty((0,) + s, device=dev) for s in self._out_shapes)

    def _step(self, n, m, H, W):
        model, S, T, C = self.model, self.streams, self.clip_len, self.channels
        w, h = self.size

        def step(x, push):
            x = x.contiguous()
            st = _st()
            _call("cvad_streams_frame_write_u8", _ptr(x), S, n, H, W, C, _ptr(self.rings), self.capacity, h, w, T, self.stride,
                  _ptr(self.cursors), _ptr(push), st)
            if m > 0:
                clips = torch.empty((S * m, C, T, h, w), device=x.device, dtype=torch.float32)
                _call("cvad_streams_clips_f32", _ptr(self.rings), S, self.capacity, h, w, C, T, self.stride, m, _ptr(self.cursors), _ptr(push),
                      1.0 / 255.0, self.reverse_channels, _ptr(clips), st)
                out = model(clips)
                out = (out[0].reshape(-1), out[1], out[2]) if C == 3 else (out.reshape(-1),)      # M-E's s.squeeze() is 0-d at S*m = 1
            else:
                out = self._empty(x.device)
            _call("cvad_streams_cursor_advance", _ptr(self.cursors), S, T, self.stride, _ptr(push), st)
            return out
        return step

    def _capture(self, n, m, frames, push):
        # warm-up runs the step for real: the rings and the cursors are restored after it, so capturing does not advance the streams
        g = GraphedStep(self._step(n, m, frames.shape[2], frames.shape[3]), (frames, push), mutated=(self.rings, self.cursors), pool=self.pool)
        cd = getattr(self.model, "causal_discovery", None)
        if cd is not None:
            # M-B's self-loop mask is cached for the latest batch size only: the next capture at another S*m replaces it, and the memory this
            # graph reads would go back to the allocator.  The graph keeps the mask it captured alive.
            g.held = list(cd._offdiag.values())
        return g

    @torch.no_grad()
    def push(self, frames, counts=None):
        """frames (S, n, H, W, C) uint8 on the model's device (C = 3, BGR, for M-B and M-E; C = 1 for M-C, which also takes (S, n, H, W)) at
        any camera size H x W; counts: S ints in [0, n], the frames each stream keeps (default n; the rows beyond a count are not read).
        Returns one (scores, first window index, adjacency, features) per stream, the records bbox:416-425 keeps per window: scores
        (w,), adjacency (w, 16, 16) and features (w, F) of its w completed windows; adjacency and features are None for M-C."""
        if frames.dim() == 4:
            frames = frames.unsqueeze(-1)
        if frames.dim() != 5:
            raise ValueError("expected (S, n, H, W, C) frames")
        if frames.dtype != torch.uint8:
            raise TypeError(f"MultiStreamClipScorer takes raw uint8 frames, got {frames.dtype}")
        if frames.shape[4] != self.channels:
            raise ValueError(f"{type(self.model).__module__}.{type(self.model).__name__} takes {self.channels}-channel frames, got {frames.shape[4]}")
        res = self._push(frames, counts, tuple(frames.shape[2:]))
        if self.channels == 1:
            return [(s, w0, None, None) for (s,), w0 in res]
        return [(s, w0, a, f) for (s, a, f), w0 in res]


class MultiStreamAutoEncoderScorer(_StreamBookkeeping):
    """Sliding-window scoring of S camera streams for M-D (``md.VideoAutoEncoder``) with one CUDA graph replay per push for all of them:
    per window the (score, reconstruction error, memory score) of ``md.calculate_anomaly_scores`` on the window's clip.

    In eval mode M-D's frame encoder and the LSTM input projection gi = W_ih latent + b_ih are per frame, so each frame is encoded once,
    however many windows contain it: the rings hold each stream's gi rows (S, capacity, 256) next to its frames (S, capacity, 4096), which
    the reconstruction error reads.  What a window needs of its own is the LSTM recurrence from a zero state at its first frame, the
    decoder and its two score terms.  ``push(frames, counts)`` runs: copy into static inputs -> ``model.encode_frames`` and the input
    projection over all S*n frames -> write each stream's kept gi rows and frames into its rings at its device cursor
    (``cvad_streams_ring_write_f32``) -> gather the gi rows of the windows each stream completed (m slots per stream,
    ``cvad_streams_window_features_f32``) -> ``ops.lstm_last`` and the eval decoder over the S*m slots -> score every slot against its
    window's frames in the frame ring and against the memory bank (``cvad_streams_md_scores_f32``; unused slots are zeros) -> advance the
    cursors.  The memory bank's fill count ``memory_ptr`` is read on the device, so ``update_memory`` and ``load_state_dict`` reach the next
    replay without a capture.

    The scores equal ``calculate_anomaly_scores`` on the window clips up to the last bits: the encoder's 2048 -> 64 layer splits its
    reduction by batch size, and here the batch is the S*n frames of a push.  Window w of a stream covers its frames w*stride + [0, clip_len)
    and is scored as soon as they have arrived (``window_count``); bbox's loop over a finished video, ``range(0, F - window, stride)``,
    stops one window earlier when (F - clip_len) % stride == 0: such a video gets one window more here, its last one.

    Counts, ``reset``, ``n_frames``, ``next_window`` and the errors are those of ``MultiStreamScorer``.  The graph key is (n, m): at most
    ceil(n / stride) + 1 graphs per push size.  Graphs share one memory pool and read the model's live tensors, so an in-place weight or
    BatchNorm-statistic update needs no capture; a replaced tensor drops them."""

    def __init__(self, model, streams, clip_len=8, stride=4, capacity=32):
        from . import md
        if not isinstance(model, md.VideoAutoEncoder):
            raise TypeError(f"MultiStreamAutoEncoderScorer scores md.VideoAutoEncoder, not {type(model).__name__}")
        super().__init__(model, streams, clip_len, stride, capacity)
        self.frame_rings = None     # (S, capacity, 64*64) fp32: the frames the reconstruction error reads

    def _new_ring(self, dev):
        self.frame_rings = torch.zeros((self.streams, self.capacity, 64 * 64), device=dev, dtype=torch.float32)
        return torch.zeros((self.streams, self.capacity, 4 * self.model.temporal_encoder.hidden_size), device=dev, dtype=torch.float32)

    def _empty(self, dev):
        return tuple(torch.empty(0, device=dev) for _ in range(3))

    def _step(self, n, m):
        model, S, T = self.model, self.streams, self.clip_len
        lstm, G, E = model.temporal_encoder, self.rings.shape[2], self.frame_rings.shape[2]

        def step(x, push):
            x = x.contiguous().reshape(S * n, 1, 64, 64)
            gi = ops.linear_act(model.encode_frames(x), lstm.weight_ih_l0, lstm.bias_ih_l0)
            st = _st()
            for src, ring, F in ((gi, self.rings, G), (x, self.frame_rings, E)):
                _call("cvad_streams_ring_write_f32", _ptr(src), S, n, F, _ptr(ring), self.capacity, T, self.stride, _ptr(self.cursors),
                      _ptr(push), st)
            if m > 0:
                win = torch.empty((S * m, T, G), device=x.device, dtype=torch.float32)
                _call("cvad_streams_window_features_f32", _ptr(self.rings), S, self.capacity, self.stride, T, G, m, _ptr(self.cursors),
                      _ptr(push), _ptr(win), st)
                z = ops.lstm_last(win, lstm.weight_hh_l0, lstm.bias_hh_l0)
                recon = model._decode_once(z, 1)
                out = tuple(torch.empty(S * m, device=x.device, dtype=torch.float32) for _ in range(3))
                mem = model.normal_memory
                _call("cvad_streams_md_scores_f32", _ptr(self.frame_rings), S, self.capacity, E, T, self.stride, m, _ptr(self.cursors),
                      _ptr(push), _ptr(recon), _ptr(z), _ptr(mem), mem.shape[0], _ptr(model.memory_ptr), mem.shape[1], *map(_ptr, out), st)
            else:
                out = self._empty(x.device)
            _call("cvad_streams_cursor_advance", _ptr(self.cursors), S, T, self.stride, _ptr(push), st)
            return out
        return step

    def _capture(self, n, m, frames, push):
        # warm-up runs the step for real: the rings and the cursors are restored after it, so capturing does not advance the streams
        return GraphedStep(self._step(n, m), (frames, push), mutated=(self.rings, self.frame_rings, self.cursors), pool=self.pool)

    @torch.no_grad()
    def push(self, frames, counts=None):
        """frames (S, n, 1, 64, 64) or (S, n, 64, 64) float32 on the model's device, in the model's input range (what
        ``calculate_anomaly_scores`` receives per clip); counts: S ints in [0, n], the frames each stream keeps (default n; the rows beyond
        a count are encoded and discarded, so they must hold finite frames).  Returns one (scores, first window index, reconstruction
        errors, memory scores) per stream, each (w,) for its w completed windows: the (scores, ..., recons, mems) of
        ``calculate_anomaly_scores``."""
        if frames.dtype != torch.float32:
            raise TypeError(f"MultiStreamAutoEncoderScorer takes float32 frames in the model's input range, got {frames.dtype}")
        if frames.dim() == 4:
            frames = frames.unsqueeze(2)
        if frames.dim() != 5 or tuple(frames.shape[2:]) != (1, 64, 64):
            raise ValueError(f"expected (S, n, 1, 64, 64) or (S, n, 64, 64) frames, got {tuple(frames.shape)}")
        return [(s, w0, r, mem) for (s, r, mem), w0 in self._push(frames, counts, ())]
