"""Low-latency inference for the per-frame (2-D backbone) models M-A and M-A0.

``FrozenBackbone`` is the bf16 tensor-core backbone of tc.py specialised to eval mode.  An eval-mode BatchNorm is a constant per-channel
affine map, so it is folded into the convolution in front of it once, at snapshot time (w' = w*s, b' = (b - running_mean)*s + beta,
s = gamma / sqrt(running_var + eps)), and every 3x3 layer is ONE launch whose tcgen05 epilogue writes relu(conv + b') straight into the
layout the next layer reads.  Per call:

  x (n,1,H,W) uint8 / fp32 --stem: space-to-depth, conv + bn1 + ReLU + max-pool--> a0 --8 x flatconv relu--> a8 --avg-pool--> (n, 6144)

11 ABI calls (the training-shaped eval path of tc._BackboneBF16 takes 36: weight packs, BatchNorm prepares, a separate apply pass that
reads every convolution output back from HBM).  The numbers differ from that path in the last bits of bf16: the folded weights are
rounded as bf16(w*s) instead of bf16(w) followed by an fp32 affine map, and the pre-activation is not rounded to bf16 before the ReLU.

``GraphedStreamingScorer`` is ``ma0.StreamingWindowScorer`` with every push of a given size replayed as one CUDA graph: the stream's
position lives in a device-side cursor, so the same graph serves every push of that size.
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


class GraphedStreamingScorer:
    """Sliding-window scoring of a frame stream, as ``ma0.StreamingWindowScorer`` (same constructor, ``push`` contract and errors), with
    each push replayed as one CUDA graph.

    A push of n frames that completes n_win windows runs: copy into a static input -> ``FrozenBackbone`` -> write the n feature rows into
    the ring at the device cursor -> gather the n_win windows -> ``model.tail`` -> advance the cursor.  Each distinct
    (n, n_win, H, W, dtype) is captured once (all graphs of one scorer share one memory pool); later pushes of it replay the graph.  The
    graphs read the model's live tensors, so in-place weight updates need nothing; a model tensor replaced by a new one (a new
    ``data_ptr``) drops the graphs, which are captured again.  Use it for a fixed chunk size and a model that is frozen or updated in
    place; a stream of ever-changing chunk sizes pays one capture per new size."""

    def __init__(self, model, clip_len=16, stride=4, capacity=256):
        if model.training:
            raise RuntimeError("GraphedStreamingScorer needs model.eval(): train-mode BatchNorm couples the frames of a batch")
        if capacity < clip_len + stride:
            raise ValueError("ring capacity must hold at least one window plus one stride of new frames")
        self.model, self.clip_len, self.stride, self.capacity = model, int(clip_len), int(stride), int(capacity)
        self.frozen = None
        self.ring = None            # (capacity, F) fp32 on the model's device
        self.cursor = None          # int64 {frames pushed, next window} on the device: what the graphs read
        self.n_frames = 0           # host mirrors of the cursor: they decide n_win and the graph key
        self.next_window = 0
        self.graphs = {}            # (n, n_win, H, W, dtype) -> GraphedStep
        self.pool = None
        self._ptrs = None

    def _model_ptrs(self):
        return [t.data_ptr() for t in list(self.model.parameters()) + list(self.model.buffers())]

    def _step(self, n, n_win):
        model, F = self.model, self.ring.shape[1]

        def step(x):
            feats = self.frozen(x)
            st = _st()
            _call("cvad_ring_write_f32", _ptr(feats), n, F, _ptr(self.ring), self.capacity, _ptr(self.cursor), st)
            if n_win > 0:
                clips = torch.empty((n_win, self.clip_len, F), device=feats.device, dtype=torch.float32)
                _call("cvad_window_features_cursor_f32", _ptr(self.ring), self.capacity, self.stride, self.clip_len, F, n_win, _ptr(self.cursor),
                      _ptr(clips), st)
                scores = model.tail(clips)["anomaly_scores"]
            else:
                scores = torch.empty(0, device=feats.device)
            _call("cvad_stream_cursor_advance", _ptr(self.cursor), n, n_win, st)
            return scores
        return step

    @torch.no_grad()
    def push(self, frames):
        """frames (n,1,H,W) float32 (normalised) or uint8 (the loader's raw frames) on the model's device -> (window scores, first window index)."""
        if frames.dim() != 4:
            raise ValueError("expected (n, 1, H, W) frames")
        n = frames.shape[0]
        if n > self.capacity - self.clip_len:
            raise ValueError("more new frames than the ring can take while it still holds an open window")
        ops._cuda(frames)
        if self.model.training:
            raise RuntimeError("GraphedStreamingScorer needs model.eval(): train-mode BatchNorm couples the frames of a batch")
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
        if self.ring is None:
            F = bb.layer4[3].out_channels * 4 * 6
            self.ring = torch.zeros((self.capacity, F), device=dev, dtype=torch.float32)
            self.cursor = torch.zeros(2, device=dev, dtype=torch.int64)
            self.pool = torch.cuda.graph_pool_handle()
        n_frames = self.n_frames + n
        n_win = 0
        if n_frames >= self.clip_len:
            n_win = (n_frames - self.clip_len) // self.stride + 1 - self.next_window
        w0 = self.next_window
        if n == 0:
            return torch.empty(0, device=dev), w0
        key = (n, max(n_win, 0), frames.shape[2], frames.shape[3], frames.dtype)
        g = self.graphs.get(key)
        if g is None:
            self.frozen._buffers(n, frames.shape[2], frames.shape[3], dev)      # allocated and zeroed outside the capture
            # warm-up runs the step for real: the ring and the cursor are restored after it, so capturing does not advance the stream
            g = self.graphs[key] = GraphedStep(self._step(n, key[1]), (frames,), mutated=(self.ring, self.cursor), pool=self.pool)
        (scores,) = g(frames)
        self.n_frames = n_frames
        self.next_window += key[1]
        return scores.clone(), w0
