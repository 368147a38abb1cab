"""M-A: the 2-D backbone + detector / tracker / GRU / VAE / causal-graph model and its train loop, on cvad_b200 kernels.

Mirrors causal_anomaly_detection.py: ``ResNetBackbone`` cad:110-158, ``SimplePedestrianDetector`` cad:160-230,
``TrajectoryTracker`` cad:232-274, ``TrajectoryEncoder`` cad:276-309, ``CausalFactorExtractor`` cad:311-352,
``CausalStructureLearner`` cad:354-398, ``DynamicsPredictor`` cad:400-426, ``EnhancedAnomalyScorer`` cad:428-502,
``CausalAnomalyDetector`` cad:508-586, ``apply_memory_efficient_training`` cad:592-607, ``train_model`` cad:609-790,
``test_model`` cad:796-835.  Module / parameter names (hence ``state_dict`` keys) and the 7-key output dict are the
reference's.  The causal branch runs as dense masked batches (5 track slots per clip + a count) instead of ragged
Python lists; the ragged lists of the output dict are materialised lazily, only if the caller indexes them.
"""
from __future__ import annotations

import collections.abc
import contextlib
import math
import os

import numpy as np
import torch
import torch.nn as nn

from . import ma_ops, ops
from .arena import FusedAdam
from .noise import DeviceNoise
from .ops import ACT_NONE, ACT_RELU, ACT_SIGMOID

SLOT_DETECTOR, SLOT_STRUCTURE, SLOT_NEVER = 1, 2, 3
TAIL_BRANCHES = os.environ.get("CVAD_TAIL_BRANCHES", "1") != "0"     # direct classifier on a second stream beside the causal branch


class ResNetBackbone(nn.Module):
    """cad:110-158 -- a plain conv/BN/ReLU stack (no residual adds), 7x7 s2 stem + maxpool + 4x2 3x3 convs + avgpool(4,6)."""

    def __init__(self, input_channels=1, output_dim=256):
        super().__init__()
        self.conv1 = nn.Conv2d(input_channels, 32, 7, stride=2, padding=3)
        self.bn1 = nn.BatchNorm2d(32)
        self.relu = nn.ReLU(inplace=True)
        self.maxpool = nn.MaxPool2d(3, stride=2, padding=1)
        self.layer1 = self._make_layer(32, 32, 2, stride=1)
        self.layer2 = self._make_layer(32, 64, 2, stride=2)
        self.layer3 = self._make_layer(64, 128, 2, stride=2)
        self.layer4 = self._make_layer(128, output_dim, 2, stride=2)
        self.avgpool = nn.AdaptiveAvgPool2d((4, 6))
        self.precision = "fp32"
        # uint8 input = the loader's raw grayscale frames (cad:89-96); they are normalised on the device as cad:1177-1179 does on the host
        self.input_mean, self.input_std = 0.5, 0.5

    @staticmethod
    def _make_layer(cin, cout, blocks, stride=1):
        layers = [nn.Conv2d(cin, cout, 3, stride=stride, padding=1), nn.BatchNorm2d(cout), nn.ReLU(inplace=True)]
        for _ in range(1, blocks):
            layers += [nn.Conv2d(cout, cout, 3, padding=1), nn.BatchNorm2d(cout), nn.ReLU(inplace=True)]
        return nn.Sequential(*layers)

    def _bn(self, h, bn):
        return ops.batchnorm_act(h, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.num_batches_tracked,
                                 ops.bn_workspace(h.device, bn.num_features), bn.training, ACT_RELU, bn.eps, bn.momentum)

    def forward(self, x):
        B, T, C, H, W = x.shape
        x = x.reshape(B * T, C, H, W)
        if x.dtype == torch.uint8 and self.precision != "bf16":
            x = ops.u8_normalize(x, self.input_mean, self.input_std)
        if self.precision == "bf16":
            from . import tc
            return tc.backbone_forward_bf16(self, x).reshape(B, T, -1)
        h = ops.conv_act(x, self.conv1.weight, self.conv1.bias, 2, 3, ACT_NONE)
        h = self._bn(h, self.bn1)
        h = ops.maxpool(h, 3, 2, 1)
        for layer in (self.layer1, self.layer2, self.layer3, self.layer4):
            for ci, bi in ((0, 1), (3, 4)):
                conv, bn = layer[ci], layer[bi]
                h = ops.conv_act(h, conv.weight, conv.bias, conv.stride, 1, ACT_NONE)
                h = self._bn(h, bn)
        h = ops.adaptive_avgpool(h, (4, 6))
        return h.reshape(B, T, -1)


def _mlp(seq, idxs, x, acts, keeps=None, ps=None, gate=None):
    """The Linear layers ``seq[idxs]`` with activations ``acts`` and dropout keep-masks ``keeps`` (probabilities ``ps``).  Layers wider
    than the fused-chain limit (the two 6144 -> 512 projections) run as GEMMs; every run of narrower layers behind them is one fused
    launch forward and one for the data-gradient chain (ops.mlp_chain).  ``gate`` (the detector's "received a gradient" flag) applies
    to the GEMM layers only: the chain is cheap enough to run on zeros."""
    layers = [(seq[li].weight, seq[li].bias, act, keeps[i] if keeps is not None else None, ps[i] if keeps is not None and keeps[i] is not None else 0.0)
              for i, (li, act) in enumerate(zip(idxs, acts))]
    h, i = x, 0
    while i < len(layers):
        din = h.shape[-1]
        j = i
        while j < len(layers) and ops.chainable(layers[i:j + 1], din):
            j += 1
        if j > i:
            h = ops.mlp_chain(h, layers[i:j])
            i = j
        else:
            w, b, act, keep, p = layers[i]
            h = ops.linear_act(h, w, b, act, keep, p, gate)
            i += 1
    return h


class SimplePedestrianDetector(nn.Module):
    """cad:160-230.  forward returns dense (box (B,T,5,4), cnt (B,T), src (B,T,5))."""

    def __init__(self, feature_dim):
        super().__init__()
        self.feature_dim = feature_dim
        self.detector_net = nn.Sequential(nn.Linear(feature_dim, 512), nn.ReLU(), nn.Dropout(0.3), nn.Linear(512, 256), nn.ReLU(),
                                          nn.Dropout(0.2), nn.Linear(256, 128), nn.ReLU(), nn.Linear(128, 64), nn.ReLU(),
                                          nn.Linear(64, 20))
        self.init_weights()

    def init_weights(self):
        with torch.no_grad():   # cad:186-192: biases start at pixel coordinates (=> saturated sigmoids, SURVEY fact 6)
            self.detector_net[-1].bias.data = torch.tensor([180, 120, 25, 50, 150, 100, 20, 45, 210, 140, 30, 55,
                                                            120, 80, 22, 48, 240, 160, 28, 52], dtype=torch.float32)

    def forward(self, features, noise, training, flag=None):
        B, T, _ = features.shape
        keeps = None
        if training:
            keeps = [noise.keep_mask("det0", (B, T, 512), 0.3, features.device), noise.keep_mask("det1", (B, T, 256), 0.2, features.device),
                     None, None, None]
        # flag: set on the device by det_decode when a real detection survives; otherwise the reference's detector output
        # is the constant fallback box, its gradient is None (SURVEY fact 6) and the backward GEMMs below switch themselves off
        raw = _mlp(self.detector_net, (0, 3, 6, 8, 10), features, (ACT_RELU, ACT_RELU, ACT_RELU, ACT_RELU, ACT_NONE), keeps,
                   (0.3, 0.2, 0, 0, 0), gate=flag)
        return ma_ops.det_decode(raw.view(B, T, 5, 4), flag)


class TrajectoryTracker(nn.Module):
    def __init__(self, max_tracks=20, reid_dim=64):
        super().__init__()
        self.max_tracks, self.reid_dim = max_tracks, reid_dim
        self.reid_net = nn.Sequential(nn.Linear(4, 32), nn.ReLU(), nn.Linear(32, reid_dim), nn.ReLU(), nn.Linear(reid_dim, reid_dim))

    def forward(self, box, cnt, flag=None):
        reid = _mlp(self.reid_net, (0, 2, 4), box, (ACT_RELU, ACT_RELU, ACT_NONE))
        return ma_ops.traj_assemble(box, reid, cnt, flag)       # (B,5,T,68), ntr (B)


class TrajectoryEncoder(nn.Module):
    def __init__(self, input_dim, latent_dim=32, hidden_dim=64):
        super().__init__()
        self.input_dim, self.latent_dim = input_dim, latent_dim
        self.gru = nn.GRU(input_dim, hidden_dim, batch_first=True, bidirectional=False)
        self.encoder = nn.Linear(hidden_dim, latent_dim)

    def last_state(self, traj, ntr):
        """traj (B,K,T,F) -> the GRU's last hidden state (B*K,64); zeros for track slots >= ntr."""
        B, K, T, F = traj.shape
        gi = ops.linear_act(traj.reshape(B * K * T, F), self.gru.weight_ih_l0, self.gru.bias_ih_l0)      # input projection GEMM
        return ma_ops.gru_last(gi.view(B * K, T, -1), self.gru.weight_hh_l0, self.gru.bias_hh_l0, ntr)

    def forward(self, traj, ntr):
        hT = self.last_state(traj, ntr)
        return ops.linear_act(hT, self.encoder.weight, self.encoder.bias).view(traj.shape[0], traj.shape[1], -1)


class CausalFactorExtractor(nn.Module):
    def __init__(self, input_dim, num_factors=6, hidden_dim=32):
        super().__init__()
        self.num_factors = num_factors
        self.encoder = nn.Sequential(nn.Linear(input_dim, hidden_dim), nn.ReLU(), nn.Linear(hidden_dim, hidden_dim), nn.ReLU())
        self.mu_head = nn.Linear(hidden_dim, num_factors)
        self.logvar_head = nn.Linear(hidden_dim, num_factors)

    def forward(self, enc, ntr, eps):
        h = _mlp(self.encoder, (0, 2), enc, (ACT_RELU, ACT_RELU))
        cur = torch.cuda.current_stream()
        side = ops.aux_stream(h.device, 2) if TAIL_BRANCHES else None
        if side is not None:
            side.wait_stream(cur)
        with (torch.cuda.stream(side) if side is not None else contextlib.nullcontext()):
            lv = ops.linear_act(h, self.logvar_head.weight, self.logvar_head.bias)       # the two heads are independent GEMMs
        mu = ops.linear_act(h, self.mu_head.weight, self.mu_head.bias)
        if side is not None:
            cur.wait_stream(side)
            lv.record_stream(cur)
        return ma_ops.reparam_kl(mu, lv, eps, ntr)               # z (B,5,6), kl (B)


class CausalStructureLearner(nn.Module):
    def __init__(self, num_factors, hidden_dim=32):
        super().__init__()
        self.num_factors = num_factors
        self.node_encoder = nn.Linear(num_factors, hidden_dim)
        self.edge_predictor = nn.Sequential(nn.Linear(hidden_dim * 2, hidden_dim), nn.ReLU(), nn.Linear(hidden_dim, 1), nn.Sigmoid())
        self.structure_params = nn.Parameter(torch.randn(num_factors, num_factors))

    def forward(self, z, ntr):
        node = ops.linear_act(z, self.node_encoder.weight, self.node_encoder.bias)          # (B,5,32)
        pair = ma_ops.pair_concat(node)                                                      # (B,5,5,64)
        e = _mlp(self.edge_predictor, (0, 2), pair, (ACT_RELU, ACT_SIGMOID))                 # (B,5,5,1)
        return ma_ops.adj_assemble(e.reshape(z.shape[0], 5, 5), ntr)                        # (B,6,6)


class DynamicsPredictor(nn.Module):
    def __init__(self, num_factors, hidden_dim=32):
        super().__init__()
        self.num_factors = num_factors
        self.dynamics_net = nn.Sequential(nn.Linear(num_factors, hidden_dim), nn.ReLU(), nn.Linear(hidden_dim, hidden_dim), nn.ReLU(),
                                          nn.Linear(hidden_dim, num_factors))

    def forward(self, z, adj):
        s = ma_ops.structured(adj, z)
        return _mlp(self.dynamics_net, (0, 2, 4), s, (ACT_RELU, ACT_RELU, ACT_NONE))


class EnhancedAnomalyScorer(nn.Module):
    """cad:428-502.  Holds the three scorers' parameters; M-A runs them inside ma_ops.causal_branch."""

    def __init__(self, num_factors):
        super().__init__()
        self.num_factors = num_factors
        self.causal_scorer = nn.Sequential(nn.Linear(num_factors * 3, 64), nn.ReLU(), nn.Dropout(0.2), nn.Linear(64, 32), nn.ReLU(),
                                           nn.Linear(32, 1), nn.Sigmoid())
        self.motion_scorer = nn.Sequential(nn.Linear(num_factors * 2, 32), nn.ReLU(), nn.Linear(32, 16), nn.ReLU(), nn.Linear(16, 1),
                                           nn.Sigmoid())
        self.temporal_scorer = nn.Sequential(nn.Linear(num_factors, 32), nn.ReLU(), nn.Linear(32, 16), nn.ReLU(), nn.Linear(16, 1),
                                             nn.Sigmoid())


class _LazyList(collections.abc.Sequence):
    """A list that is built (with one device->host sync) only when somebody indexes it."""

    def __init__(self, build):
        self._build, self._items = build, None

    def _get(self):
        if self._items is None:
            self._items = self._build()
        return self._items

    def __getitem__(self, i):
        return self._get()[i]

    def __len__(self):
        return len(self._get())


class CausalAnomalyDetector(nn.Module):
    """cad:508-586.  forward((B,T,1,H,W)) -> dict with the reference's 7 keys (+ 'dense': the batched tensors)."""

    def __init__(self, num_factors=6, reid_dim=64):
        super().__init__()
        self.backbone = ResNetBackbone(input_channels=1, output_dim=256)
        self.detector = SimplePedestrianDetector(256 * 4 * 6)
        self.tracker = TrajectoryTracker(reid_dim=reid_dim)
        self.traj_encoder = TrajectoryEncoder(4 + reid_dim, latent_dim=32)
        self.causal_extractor = CausalFactorExtractor(32, num_factors=num_factors)
        self.structure_learner = CausalStructureLearner(num_factors)
        self.dynamics_predictor = DynamicsPredictor(num_factors)
        self.anomaly_scorer = EnhancedAnomalyScorer(num_factors)
        self.direct_classifier = nn.Sequential(nn.Linear(256 * 4 * 6, 512), nn.ReLU(), nn.Dropout(0.3), nn.Linear(512, 256), nn.ReLU(),
                                               nn.Dropout(0.2), nn.Linear(256, 128), nn.ReLU(), nn.Linear(128, 64), nn.ReLU(),
                                               nn.Linear(64, 2), nn.Softmax(dim=-1))
        self.noise = DeviceNoise()
        self.flags = None            # gradient-arena header (set by the trainer): activity flags for "grad is None" groups

    def set_precision(self, precision: str):
        assert precision in ("fp32", "bf16")
        self.backbone.precision = precision
        return self

    def optimizer_slots(self):
        """Parameters that may legitimately receive no gradient in a step (torch leaves .grad None, AdamW skips them)."""
        slots = {}
        for p in self.detector.parameters():
            slots[id(p)] = SLOT_DETECTOR
        for p in list(self.structure_learner.node_encoder.parameters()) + list(self.structure_learner.edge_predictor.parameters()):
            slots[id(p)] = SLOT_STRUCTURE
        slots[id(self.structure_learner.structure_params)] = SLOT_NEVER
        return slots

    def causal_branch_params(self):
        """The 40 weight / bias tensors of the causal branch behind the GRU, in the order of ma_ops.causal_branch."""
        sc = self.anomaly_scorer
        layers = [self.traj_encoder.encoder, self.causal_extractor.encoder[0], self.causal_extractor.encoder[2], self.causal_extractor.mu_head,
                  self.causal_extractor.logvar_head, self.structure_learner.node_encoder, self.structure_learner.edge_predictor[0],
                  self.structure_learner.edge_predictor[2], *(self.dynamics_predictor.dynamics_net[i] for i in (0, 2, 4)),
                  *(sc.causal_scorer[i] for i in (0, 3, 5)), *(sc.motion_scorer[i] for i in (0, 2, 4)),
                  *(sc.temporal_scorer[i] for i in (0, 2, 4))]
        return [t for lin in layers for t in (lin.weight, lin.bias)]

    def forward(self, video_frames, feature_cut=None):
        """``feature_cut``: a list that receives ``(features, leaf)`` -- the autograd graph is cut behind the backbone (``leaf`` is a
        detached copy the rest of the model consumes), so a trainer can run the tail's backward first and the backbone's backward
        (``features.backward(leaf.grad)``) as a separate, later stage while the tail's gradients are already being all-reduced."""
        features = self.backbone(video_frames)
        if feature_cut is not None and features.requires_grad:
            leaf = features.detach().requires_grad_(True)
            feature_cut.append((features, leaf))
            features = leaf
        return self.tail(features)

    def tail(self, features):
        """Everything behind the backbone: features (B,T,6144) -> the output dict (cad:546-586).  In eval mode a frame's features do not
        depend on its clip, which is what ma0.StreamingWindowScorer builds on."""
        B, T, _ = features.shape
        dev = features.device
        f_det = self.flags[SLOT_DETECTOR:SLOT_DETECTOR + 1] if self.flags is not None else None
        f_str = self.flags[SLOT_STRUCTURE:SLOT_STRUCTURE + 1] if self.flags is not None else None
        # The direct classifier (cad:525-538, 568-571) depends on the features only: it runs on a second stream beside the dependent
        # launches of the detector, tracker, GRU and causal branch (autograd replays the fork in the backward: the classifier's
        # data-gradient chain and its 6144-wide GEMM run beside the causal branch's); in a captured step the two become parallel branches
        # of the graph.
        cur = torch.cuda.current_stream()
        side = ops.aux_stream(dev, 1) if TAIL_BRANCHES else None
        keeps = None
        if self.training:
            keeps = [self.noise.keep_mask("cls0", (B, 512), 0.3, dev), self.noise.keep_mask("cls1", (B, 256), 0.2, dev), None, None, None]
        # (a view taken on THIS stream: its backward node -- no kernel -- hands the branch's gradient to the features' accumulation on
        # the stream the features live on)
        fsrc = features.view_as(features) if side is not None else features
        if side is not None:
            side.wait_stream(cur)
        with (torch.cuda.stream(side) if side is not None else contextlib.nullcontext()):
            pooled = ops.mean_mid(fsrc)
            logits = _mlp(self.direct_classifier, (0, 3, 6, 8, 10), pooled, (ACT_RELU, ACT_RELU, ACT_RELU, ACT_RELU, ACT_NONE), keeps,
                          (0.3, 0.2, 0, 0, 0))
            direct = ma_ops.softmax_rows(logits)
        box, cnt, _src = self.detector(features, self.noise, self.training, f_det)
        traj, ntr = self.tracker(box, cnt, f_str)
        hT = self.traj_encoder.last_state(traj, ntr)
        eps = self.noise.normal("eps", (B, 5, 6), dev)          # drawn in eval mode too (cad:328-331)
        keep0 = self.noise.keep_mask("scorer0", (B, 64), 0.2, dev) if self.training else None
        # everything from the GRU's last state to (z, kl, adj, causal score): one kernel forward, one backward
        z, kl, adj, causal = ma_ops.causal_branch(hT, ntr, eps, keep0, self.causal_branch_params())
        if side is not None:
            cur.wait_stream(side)
            direct.record_stream(cur)
        final = ops.lincomb2(causal, 0.6, direct, 1, 0.4)       # cad:574
        dense = {"causal_factors": z, "adjacency_matrices": adj, "kl_losses": kl, "detections": box, "det_counts": cnt,
                 "n_tracks": ntr, "features": features}

        def ragged_factors():
            n = ntr.tolist()
            return [z[b, :n[b]] for b in range(B)]

        def ragged_dets():
            c = cnt.tolist()
            return [[box[b, t, :c[b][t]] for t in range(T)] for b in range(B)]

        return {
            "anomaly_scores": final,
            "causal_factors": _LazyList(ragged_factors),
            "adjacency_matrices": _LazyList(lambda: [adj[b] for b in range(B)]),
            "kl_losses": _LazyList(lambda: [kl[b] for b in range(B)]),
            "detections": _LazyList(ragged_dets),
            "direct_predictions": direct,
            "causal_anomaly_scores": causal,
            "dense": dense,
        }


def apply_memory_efficient_training(model, verbose=False):
    """cad:592-607: freeze the stem (backbone.conv1 / backbone.bn1)."""
    for name, param in model.named_parameters():
        if "backbone.conv1" in name or "backbone.bn1" in name:
            param.requires_grad = False
    if verbose:
        total = sum(p.numel() for p in model.parameters())
        trainable = sum(p.numel() for p in model.parameters() if p.requires_grad)
        print(f"Total parameters: {total:,}\nTrainable parameters: {trainable:,}\nFrozen parameters: {total - trainable:,}")
    return model


class MATrainer:
    """The loop body of cad:637-693 as an object: 4-term fused loss, clip 1.0, AdamW(lr 3e-4, wd 1e-5), cosine schedule."""

    def __init__(self, model, device, num_epochs=20, lr=3e-4, precision="fp32", dp=None):
        self.device = torch.device(device) if not isinstance(device, torch.device) else device
        if self.device.type != "cuda":
            raise RuntimeError("M-A trainer (cvad_b200) requires a CUDA device; there is no CPU fallback")
        self.model = apply_memory_efficient_training(model).to(self.device)
        self.model.set_precision(precision)
        params = [p for p in self.model.parameters() if p.requires_grad]
        self.optimizer = FusedAdam(params, lr=lr, weight_decay=1e-5, eps=1e-8, decoupled=True, clip_mode=1, max_norm=1.0, nan_mode=1,
                                   slots=self.model.optimizer_slots())
        self.model.flags = self.optimizer.arena.header
        self.scheduler = torch.optim.lr_scheduler.CosineAnnealingLR(self.optimizer, T_max=num_epochs)
        self.dp = dp
        if dp is not None:
            dp.attach(self.optimizer)
            # arena order = model.parameters() order: backbone first.  Everything from the first non-backbone tensor on is "early".
            arena = self.optimizer.arena
            backbone_ids = {id(p) for p in self.model.backbone.parameters()}
            first = next((o for p, o in zip(arena.params, arena.offsets) if id(p) not in backbone_ids), arena.total)
            dp.set_split(first)

    def loss_on_device(self, outputs, labels):
        d = outputs["dense"]
        return ops.ma_loss(outputs["direct_predictions"], outputs["anomaly_scores"], outputs["causal_anomaly_scores"], d["kl_losses"],
                           labels, self.optimizer.arena.header[0:1])

    def forward_backward(self, videos, labels):
        self.optimizer.zero_grad()
        outputs = self.model(videos)
        loss, comp = self.loss_on_device(outputs, labels)
        with ops.param_grad_overlap():          # weight/bias-gradient kernels of the dense tail run beside the data-gradient chain
            loss.backward()
        return comp, outputs

    def train_step(self, videos, labels):
        comp, outputs = self.forward_backward(videos, labels)
        self.optimizer.step()
        return comp, outputs

    def mutated_tensors(self):
        """Everything a train step changes in place (what a CUDA-graph warm-up has to restore)."""
        a = self.optimizer.arena
        return [a.p, a.m, a.v, a.state] + [b for b in self.model.buffers()]

    def graphed_train_step(self, videos, labels):
        """One CUDA graph for zero_grad + forward + loss + backward (+ all-reduce) + clip/AdamW on this batch shape.
        Returns a callable ``(videos, labels) -> (loss components (5,), anomaly_scores (B,))``."""
        from .graphs import graphed_optimizer_step

        if self.dp is None:
            def fwd_bwd(x, y):
                comp, out = self.forward_backward(x, y)
                return comp, out["anomaly_scores"]
            return graphed_optimizer_step(self.optimizer, fwd_bwd, (videos, labels), self.mutated_tensors())

        # data parallel: the backward is captured in two stages so that the gradients of everything behind the backbone (26 of the 31 MB
        # of the arena) are all-reduced over NVLink while the backbone's backward -- 45 % of the step -- is still running
        cut = []

        def fwd_bwd(x, y):
            self.optimizer.zero_grad()
            cut.clear()
            outputs = self.model(x, feature_cut=cut)
            loss, comp = self.loss_on_device(outputs, y)
            with ops.param_grad_overlap():
                loss.backward()
            return comp, outputs["anomaly_scores"]

        def backbone_backward():
            feats, leaf = cut[0]
            feats.backward(leaf.grad)

        return graphed_optimizer_step(self.optimizer, fwd_bwd, (videos, labels), self.mutated_tensors(), late_backward=backbone_backward)

    @torch.no_grad()
    def eval_step(self, videos, labels):
        outputs = self.model(videos)
        _, comp = self.loss_on_device(outputs, labels)
        return comp, outputs


def train_model(model, train_loader, val_loader, num_epochs=20, lr=3e-4, device="cuda", precision="bf16", verbose=True):
    """cad:609-790.  Returns (model, train_losses, val_losses).  Mixed precision = bf16 operands / fp32 accumulation on the
    tensor cores (the reference uses fp16 autocast + GradScaler, cad:621,645; no loss scaling is needed for bf16)."""
    tr = MATrainer(model, device, num_epochs, lr, precision)
    train_losses, val_losses = [], []
    for epoch in range(num_epochs):
        tr.model.train()
        acc = torch.zeros(2, device=tr.device)
        for videos, labels in train_loader:
            videos = videos.to(tr.device, non_blocking=True)
            labels = labels.to(tr.device, non_blocking=True)
            comp, _ = tr.train_step(videos, labels)
            ok = torch.isfinite(comp[0]).float()
            acc[0] += torch.nan_to_num(comp[0]) * ok
            acc[1] += 1
        tr.model.eval()
        vacc = torch.zeros(4, device=tr.device)
        for videos, labels in val_loader:
            videos = videos.to(tr.device, non_blocking=True)
            labels = labels.to(tr.device, non_blocking=True)
            comp, out = tr.eval_step(videos, labels)
            vacc[0] += comp[0]
            vacc[1] += 1
            vacc[2] += (out["direct_predictions"].argmax(dim=1) == labels).sum()
            vacc[3] += labels.numel()
        tr.scheduler.step()
        a, v = acc.tolist(), vacc.tolist()
        train_losses.append(a[0] / max(a[1], 1))
        val_losses.append(v[0] / max(v[1], 1))
        if verbose:
            print(f"Epoch {epoch + 1}/{num_epochs}, Train Loss: {train_losses[-1]:.6f}, Val Loss: {val_losses[-1]:.6f}, "
                  f"Val Accuracy: {v[2] / max(v[3], 1):.4f}")
    return tr.model, train_losses, val_losses


@torch.no_grad()
def test_model(model, test_loader, device="cuda"):
    """cad:796-835: returns (scores, labels, list of output dicts)."""
    model.eval()
    dev = torch.device(device)
    scores, labels_all, outs = [], [], []
    for videos, labels in test_loader:
        out = model(videos.to(dev))
        scores.append(out["anomaly_scores"])
        labels_all.extend(np.asarray(labels).tolist())
        outs.append(out)
    return torch.cat(scores).cpu().numpy(), np.array(labels_all), outs
