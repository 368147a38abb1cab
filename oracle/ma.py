"""Oracle (TEST INFRASTRUCTURE) for M-A: the 2-D backbone + detector/tracker/GRU/VAE/graph model.

Follows causal_anomaly_detection.py (cad): backbone cad:110-158, detector cad:160-230,
tracker cad:232-274, trajectory encoder cad:276-309, factor extractor cad:311-352,
structure learner cad:354-398, dynamics cad:400-426, scorer cad:428-502, model cad:508-586,
4-term loss cad:649-662.

It is written as a dense, masked, batched restatement (tracks padded to 5 per clip with a
per-clip track count) rather than the reference's ragged Python lists; tools/make_golden.py
proves the two agree, including on inputs where the detector emits 1..5 valid boxes.
All noise is explicit: ``eps`` (B,5,6) for the reparameterisation (drawn in eval mode too,
cad:328-331) and dropout keep-masks in ``keep``.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

BN_EPS, BN_MOM = 1e-5, 0.1
MAXDET = 5
NF = 6


def _bn2d(h, P, name, train, new_stats):
    w, b = P[name + ".weight"], P[name + ".bias"]
    if train:
        mean = h.mean(dim=(0, 2, 3))
        var = h.var(dim=(0, 2, 3), unbiased=False)
        n = h.numel() // h.shape[1]
        if new_stats is not None:
            new_stats[name + ".running_mean"] = (1 - BN_MOM) * P[name + ".running_mean"] + BN_MOM * mean.detach()
            new_stats[name + ".running_var"] = (1 - BN_MOM) * P[name + ".running_var"] + BN_MOM * var.detach() * n / max(n - 1, 1)
            new_stats[name + ".num_batches_tracked"] = P[name + ".num_batches_tracked"] + 1
    else:
        mean, var = P[name + ".running_mean"], P[name + ".running_var"]
    sh = (1, -1, 1, 1)
    return (h - mean.view(sh)) / torch.sqrt(var.view(sh) + BN_EPS) * w.view(sh) + b.view(sh)


def backbone(P, x, train=False, new_stats=None):
    """x (B,T,1,H,W) -> (B,T,6144).  cad:141-158 (a plain conv/BN/ReLU stack: no residual adds)."""
    B, T, C, H, W = x.shape
    h = x.reshape(B * T, C, H, W)
    h = F.conv2d(h, P["backbone.conv1.weight"], P["backbone.conv1.bias"], stride=2, padding=3)
    h = F.relu(_bn2d(h, P, "backbone.bn1", train, new_stats))
    h = F.max_pool2d(h, 3, stride=2, padding=1)
    for layer, stride in ((1, 1), (2, 2), (3, 2), (4, 2)):
        for ci, bi, s in ((0, 1, stride), (3, 4, 1)):
            pre = f"backbone.layer{layer}."
            h = F.conv2d(h, P[pre + f"{ci}.weight"], P[pre + f"{ci}.bias"], stride=s, padding=1)
            h = F.relu(_bn2d(h, P, pre + str(bi), train, new_stats))
    h = F.adaptive_avg_pool2d(h, (4, 6))
    return h.reshape(B, T, -1)


def _mlp(P, prefix, idxs, x, acts, keeps=None, ps=None):
    """Sequential of Linear layers at ``idxs`` with activation names in ``acts``;
    ``keeps[i]`` (or None) is the dropout keep-mask applied after activation i with prob ps[i]."""
    h = x
    for i, (li, act) in enumerate(zip(idxs, acts)):
        h = F.linear(h, P[f"{prefix}.{li}.weight"], P[f"{prefix}.{li}.bias"])
        if act == "relu":
            h = F.relu(h)
        elif act == "sigmoid":
            h = torch.sigmoid(h)
        if keeps is not None and keeps[i] is not None:
            h = h * keeps[i] * (1.0 / (1.0 - ps[i]))
    return h


def detect(P, feats, train, keep):
    """cad:194-230.  Returns boxes (B,T,5,4) compacted (valid first, original order; fallback
    row when none valid), counts (B,T) int64."""
    B, T, _ = feats.shape
    keeps = [keep.get("det0"), keep.get("det1"), None, None, None] if train else None
    raw = _mlp(P, "detector.detector_net", (0, 3, 6, 8, 10), feats, ("relu", "relu", "relu", "relu", None),
               keeps, (0.3, 0.2, 0, 0, 0)).view(B, T, MAXDET, 4)
    scale = torch.tensor([360.0, 240.0, 80.0, 120.0])
    off = torch.tensor([0.0, 0.0, 15.0, 25.0])
    box = torch.sigmoid(raw) * scale + off                                  # cad:201-204
    lo = torch.tensor([10.0, 10.0, 10.0, 20.0])
    hi = torch.tensor([350.0, 230.0, 100.0, 150.0])
    valid = ((box >= lo) & (box <= hi)).all(dim=-1)                         # cad:217-218
    cnt = valid.sum(dim=-1)
    out = torch.zeros_like(box)
    fallback = torch.tensor([180.0, 120.0, 30.0, 60.0])                      # cad:225
    for b in range(B):
        for t in range(T):
            sel = box[b, t][valid[b, t]]
            if sel.shape[0] == 0:
                out[b, t, 0] = fallback
            else:
                out[b, t, : sel.shape[0]] = sel
    cnt = torch.clamp(cnt, min=1)
    return out, cnt


def gru_last(P, x):
    """nn.GRU(68->64, batch_first) last hidden state; x (N,T,68).  cad:284, 298-299."""
    Wi, Wh = P["traj_encoder.gru.weight_ih_l0"], P["traj_encoder.gru.weight_hh_l0"]
    bi, bh = P["traj_encoder.gru.bias_ih_l0"], P["traj_encoder.gru.bias_hh_l0"]
    N, T, _ = x.shape
    Hd = Wh.shape[1]
    h = torch.zeros(N, Hd, dtype=x.dtype)
    for t in range(T):
        gi = F.linear(x[:, t], Wi, bi)
        gh = F.linear(h, Wh, bh)
        r = torch.sigmoid(gi[:, :Hd] + gh[:, :Hd])
        z = torch.sigmoid(gi[:, Hd:2 * Hd] + gh[:, Hd:2 * Hd])
        n = torch.tanh(gi[:, 2 * Hd:] + r * gh[:, 2 * Hd:])
        h = (1 - z) * n + z * h
    return h


def ma_forward(P: dict, x: torch.Tensor, eps: torch.Tensor, train: bool = False, keep: dict | None = None,
               new_stats: dict | None = None):
    """x (B,T,1,H,W) -> dict mirroring cad:578-586 with dense tensors:
    anomaly_scores (B,), causal_factors (B,5,6), adjacency_matrices (B,6,6), kl_losses (B,),
    detections (B,T,5,4) + det_counts (B,T), n_tracks (B,), direct_predictions (B,2),
    causal_anomaly_scores (B,)."""
    feats = backbone(P, x, train, new_stats)
    return ma_tail(P, feats, eps, train, keep)


def ma_tail(P: dict, feats: torch.Tensor, eps: torch.Tensor, train: bool = False, keep: dict | None = None):
    """Everything behind the backbone: feats (B,T,6144) -> the dict of ``ma_forward``.  Runs in the features' dtype (float64 included:
    the fp64 reference of the causal branch's kernels)."""
    keep = keep or {}
    B, T, _ = feats.shape
    box, cnt = detect(P, feats, train, keep)
    ntr = cnt.max(dim=1).values                                              # tracks per clip, cad:260
    kidx = torch.arange(MAXDET)
    row_ok = (kidx.view(1, 1, -1) < cnt.unsqueeze(-1)).float().unsqueeze(-1)  # (B,T,5,1)
    reid = _mlp(P, "tracker.reid_net", (0, 2, 4), box, ("relu", "relu", None))
    traj = torch.cat([box, reid], dim=-1) * row_ok                           # zero padding rows, cad:264-266
    trk_ok = (kidx.view(1, -1) < ntr.unsqueeze(-1)).float()                  # (B,5)
    hT = gru_last(P, traj.permute(0, 2, 1, 3).reshape(B * MAXDET, T, -1))
    enc = F.linear(hT, P["traj_encoder.encoder.weight"], P["traj_encoder.encoder.bias"]).view(B, MAXDET, -1)
    h = _mlp(P, "causal_extractor.encoder", (0, 2), enc, ("relu", "relu"))
    mu = F.linear(h, P["causal_extractor.mu_head.weight"], P["causal_extractor.mu_head.bias"])
    lv = F.linear(h, P["causal_extractor.logvar_head.weight"], P["causal_extractor.logvar_head.bias"])
    z = mu + eps * torch.exp(0.5 * lv)                                       # cad:328-331
    klrow = -0.5 * (1 + lv - mu.pow(2) - lv.exp()).sum(dim=-1)               # cad:344
    kl = (klrow * trk_ok).sum(dim=1) / ntr
    # structure learner: rows/cols index TRACKS (cad:382-387), matrix is num_factors x num_factors
    node = F.linear(z, P["structure_learner.node_encoder.weight"], P["structure_learner.node_encoder.bias"])
    adj = torch.zeros(B, NF, NF, dtype=feats.dtype)
    pair = torch.cat([node.unsqueeze(2).expand(B, MAXDET, MAXDET, -1), node.unsqueeze(1).expand(B, MAXDET, MAXDET, -1)], dim=-1)
    e = _mlp(P, "structure_learner.edge_predictor", (0, 2), pair, ("relu", "sigmoid")).squeeze(-1)   # (B,5,5)
    emask = trk_ok.unsqueeze(2) * trk_ok.unsqueeze(1) * (1 - torch.eye(MAXDET))
    adj[:, :MAXDET, :MAXDET] = e * emask
    # dynamics: (adj @ z^T)^T per track, cad:420-421 -- adj multiplies the FACTOR axis
    structured = torch.einsum("bij,bkj->bki", adj, z)
    pred = _mlp(P, "dynamics_predictor.dynamics_net", (0, 2, 4), structured, ("relu", "relu", None))
    w = (trk_ok / ntr.unsqueeze(-1)).unsqueeze(-1)
    cur = (z * w).sum(dim=1)                                                 # mean over tracks, cad:470-472
    prd = (pred * w).sum(dim=1)
    diff = (cur - prd).abs()
    keeps = [keep.get("scorer0"), None, None] if train else None
    cs = _mlp(P, "anomaly_scorer.causal_scorer", (0, 3, 5), torch.cat([cur, prd, diff], -1),
              ("relu", "relu", "sigmoid"), keeps, (0.2, 0, 0))
    ms = _mlp(P, "anomaly_scorer.motion_scorer", (0, 2, 4), torch.cat([cur, prd], -1), ("relu", "relu", "sigmoid"))
    ts = _mlp(P, "anomaly_scorer.temporal_scorer", (0, 2, 4), cur, ("relu", "relu", "sigmoid"))
    causal = (0.5 * cs + 0.3 * ms + 0.2 * ts).squeeze(-1)                    # cad:497
    pooled = feats.mean(dim=1)                                               # cad:568
    keeps = [keep.get("cls0"), keep.get("cls1"), None, None, None] if train else None
    logits = _mlp(P, "direct_classifier", (0, 3, 6, 8, 10), pooled, ("relu", "relu", "relu", "relu", None),
                  keeps, (0.3, 0.2, 0, 0, 0))
    direct = torch.softmax(logits, dim=-1)                                   # cad:537
    final = 0.6 * causal + 0.4 * direct[:, 1]                                # cad:574
    return {
        "anomaly_scores": final, "causal_factors": z, "adjacency_matrices": adj, "kl_losses": kl,
        "detections": box, "det_counts": cnt, "n_tracks": ntr, "direct_predictions": direct,
        "causal_anomaly_scores": causal, "features": feats,
    }


def ma_loss(out: dict, labels: torch.Tensor):
    """cad:649-662.  CrossEntropy is applied to the already-softmaxed probabilities (double softmax)."""
    y = labels.to(out["anomaly_scores"].dtype)
    ce = F.cross_entropy(out["direct_predictions"], labels)
    mse_final = F.mse_loss(out["anomaly_scores"], y)
    kl = out["kl_losses"]
    klm = torch.where(torch.isfinite(kl), kl, torch.zeros_like(kl)).sum() / kl.shape[0]   # cad:653-654
    mse_causal = F.mse_loss(out["causal_anomaly_scores"], y)
    total = 0.4 * ce + 0.3 * mse_final + 0.2 * mse_causal + 0.1 * klm
    return total, {"classification": float(ce.detach()), "anomaly": float(mse_final.detach()), "causal": float(mse_causal.detach()), "kl": float(klm.detach())}
