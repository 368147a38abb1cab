"""M-D: the convolutional autoencoder + LSTM + normal-pattern memory bank of causal_anomaly_detection1.py, on cvad_b200 kernels.

Mirrors ``VideoAutoEncoder`` cad1:124-321 (module / parameter / buffer names, hence ``state_dict`` keys incl.
``normal_memory``, ``memory_ptr``, ``temperature``), ``reconstruction_loss`` cad1:340-344, ``calculate_anomaly_scores``
cad1:526-564 and the loop body of ``train_model`` cad1:346-440 (Adam lr, L2 weight decay 1e-6, clip 0.1, skip on a
non-finite loss or gradient -- decided on the device instead of through per-parameter host syncs).

Differences in execution, not in results:
* the frame encoder runs once over all B*T frames (time-major) instead of T Python iterations; its BatchNorms keep the
  reference's per-time-step batch statistics and T sequential running-statistics updates (``ops.batchnorm_act``);
* the decoder, which the reference runs T times on the SAME sequence feature (cad1:254-257), runs once; ``reconstructed``
  is that frame viewed T times, the loss kernel sums the T targets' gradients, and the decoder BatchNorms' running
  statistics receive their T-1 further (identical) updates in closed form.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn

from . import ops
from .arena import FusedAdam
from .ops import ACT_LEAKY01, ACT_NONE, ACT_SIGMOID, ACT_TANH


def init_weights(m):
    """cad1:29-42."""
    if isinstance(m, (nn.Conv2d, nn.ConvTranspose2d)):
        nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="leaky_relu")
        if m.bias is not None:
            nn.init.constant_(m.bias, 0)
    elif isinstance(m, nn.Linear):
        nn.init.xavier_normal_(m.weight, gain=0.5)
        if m.bias is not None:
            nn.init.constant_(m.bias, 0)
    elif isinstance(m, nn.BatchNorm2d):
        nn.init.constant_(m.weight, 1)
        nn.init.constant_(m.bias, 0)


def _bn(h, bn, groups=1):
    return ops.batchnorm_act(h, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.num_batches_tracked,
                             ops.bn_workspace(h.device, bn.num_features), bn.training, ACT_LEAKY01, bn.eps, bn.momentum, groups)


class VideoAutoEncoder(nn.Module):
    """cad1:124-321.  forward((B,T,1,64,64)) -> {'reconstructed', 'sequence_feature', 'frame_features', 'anomaly_score'}."""

    def __init__(self, input_channels=1, latent_dim=64):
        super().__init__()
        if latent_dim != 64:
            raise ValueError("the LSTM kernel implements the reference's latent_dim = 64 (cad1:125)")
        L = nn.LeakyReLU(0.1, inplace=True)
        self.encoder = nn.Sequential(
            nn.Conv2d(input_channels, 32, 4, stride=2, padding=1), nn.BatchNorm2d(32), L,
            nn.Conv2d(32, 64, 4, stride=2, padding=1), nn.BatchNorm2d(64), nn.LeakyReLU(0.1, inplace=True),
            nn.Conv2d(64, 128, 4, stride=2, padding=1), nn.BatchNorm2d(128), nn.LeakyReLU(0.1, inplace=True),
            nn.Conv2d(128, 128, 4, stride=2, padding=1), nn.BatchNorm2d(128), nn.LeakyReLU(0.1, inplace=True),
            nn.Flatten(), nn.Linear(128 * 4 * 4, latent_dim), nn.Tanh())
        self.decoder = nn.Sequential(
            nn.Linear(latent_dim, 128 * 4 * 4), nn.LeakyReLU(0.1, inplace=True), nn.Unflatten(1, (128, 4, 4)),
            nn.ConvTranspose2d(128, 128, 4, stride=2, padding=1), nn.BatchNorm2d(128), nn.LeakyReLU(0.1, inplace=True),
            nn.ConvTranspose2d(128, 64, 4, stride=2, padding=1), nn.BatchNorm2d(64), nn.LeakyReLU(0.1, inplace=True),
            nn.ConvTranspose2d(64, 32, 4, stride=2, padding=1), nn.BatchNorm2d(32), nn.LeakyReLU(0.1, inplace=True),
            nn.ConvTranspose2d(32, input_channels, 4, stride=2, padding=1), nn.Sigmoid())
        self.temporal_encoder = nn.LSTM(input_size=latent_dim, hidden_size=latent_dim, num_layers=1, batch_first=True, dropout=0.0)
        self.register_buffer("normal_memory", torch.zeros(500, latent_dim))
        self.register_buffer("memory_ptr", torch.zeros(1, dtype=torch.long))
        self.memory_size = 500
        self.apply(init_weights)
        self.register_buffer("temperature", torch.tensor(1.0))
        self._ptr_host = None          # host mirror of memory_ptr (the reference reads it with int(), a sync, every call)

    # ---- memory bank (cad1:201-219)
    def _ptr(self) -> int:
        if self._ptr_host is None:
            self._ptr_host = int(self.memory_ptr)
        return self._ptr_host

    def load_state_dict(self, *a, **k):
        out = super().load_state_dict(*a, **k)
        self._ptr_host = None
        return out

    @torch.no_grad()
    def update_memory(self, features):
        features = features.detach()
        bs, ptr = features.shape[0], self._ptr()
        if ptr + bs <= self.memory_size:
            self.normal_memory[ptr:ptr + bs] = features
            new = (ptr + bs) % self.memory_size
        else:
            remaining = self.memory_size - ptr
            self.normal_memory[ptr:] = features[:remaining]
            self.normal_memory[:bs - remaining] = features[remaining:]
            new = bs - remaining
        self._ptr_host = new
        self.memory_ptr.fill_(new)

    # ---- encoder / decoder
    def encode_frames(self, x, groups=1):
        """The frame encoder (cad1:227-234): x (N, C, 64, 64) -> latents (N, 64).  In train mode the BatchNorms take their batch
        statistics over each of ``groups`` equal, contiguous blocks of frames (one time step each); in eval mode a frame's latent depends
        on that frame alone."""
        e = self.encoder
        h = x
        for ci in (0, 3, 6, 9):
            conv, bn = e[ci], e[ci + 1]
            h = ops.conv_act(h, conv.weight, conv.bias, 2, 1, ACT_NONE)
            h = _bn(h, bn, groups)
        return ops.linear_act(h.reshape(x.shape[0], -1), e[13].weight, e[13].bias, ACT_TANH)

    def encode_sequence(self, frames):
        B, T, C, H, W = frames.shape
        groups = T if self.training else 1           # per-time-step batch statistics in train mode (cad1:227-231)
        h = frames.transpose(0, 1).reshape(T * B, C, H, W)      # time-major: each step's B frames are contiguous
        lat = self.encode_frames(h, groups)                                                       # (T*B, 64)
        frame_features = lat.reshape(T, B, -1).transpose(0, 1)                                    # (B, T, 64) view
        lstm = self.temporal_encoder
        gi = ops.linear_act(frame_features.reshape(B * T, -1), lstm.weight_ih_l0, lstm.bias_ih_l0).reshape(B, T, -1)
        sequence_feature = ops.lstm_last(gi, lstm.weight_hh_l0, lstm.bias_hh_l0)
        return sequence_feature, frame_features

    def _decode_once(self, z, repeats):
        d = self.decoder
        h = ops.linear_act(z, d[0].weight, d[0].bias, ACT_LEAKY01).reshape(z.shape[0], 128, 4, 4)
        for ci in (3, 6, 9):
            ct, bn = d[ci], d[ci + 1]
            h = ops.channel_bias_act(ops.conv_transpose2d(h, ct.weight, 2, 1), ct.bias, ACT_NONE)
            if bn.training and repeats > 1:
                rm0, rv0 = bn.running_mean.clone(), bn.running_var.clone()
            h = _bn(h, bn)
            if bn.training and repeats > 1:
                # the reference calls this BatchNorm `repeats` times on identical input: apply the remaining updates
                with torch.no_grad():
                    m = bn.momentum
                    bm = (bn.running_mean - (1 - m) * rm0) / m
                    bv = (bn.running_var - (1 - m) * rv0) / m
                    k = (1 - m) ** (repeats - 1)
                    bn.running_mean.mul_(k).add_(bm * (1 - k))
                    bn.running_var.mul_(k).add_(bv * (1 - k))
                    bn.num_batches_tracked += repeats - 1
        ct = d[12]
        return ops.channel_bias_act(ops.conv_transpose2d(h, ct.weight, 2, 1), ct.bias, ACT_SIGMOID)

    def decode_sequence(self, sequence_feature, sequence_length):
        frame = self._decode_once(sequence_feature, sequence_length)                    # (B, C, H, W)
        out = frame.unsqueeze(1).expand(-1, sequence_length, -1, -1, -1)
        out._cvad_base = frame          # lets the loss / scoring kernels skip the T-fold broadcast (and its autograd)
        return out

    def compute_anomaly_score(self, sequence_feature):
        return ops.memory_score(sequence_feature, self.normal_memory, self._ptr())

    def forward(self, frames):
        if frames.dim() != 5:
            raise ValueError(f"expected (B,T,C,H,W) frames, got {tuple(frames.shape)}")
        T = frames.shape[1]
        sequence_feature, frame_features = self.encode_sequence(frames)
        reconstructed = self.decode_sequence(sequence_feature, T)
        return {"reconstructed": reconstructed, "sequence_feature": sequence_feature, "frame_features": frame_features,
                "anomaly_score": self.compute_anomaly_score(sequence_feature)}


def _base_frame(reconstructed):
    """The single decoded frame behind a broadcast ``reconstructed`` (stride 0 over T), else None."""
    return getattr(reconstructed, "_cvad_base", None)


def reconstruction_loss(original, reconstructed, flag=None):
    """cad1:340-344 (MSE).  A NaN/Inf loss raises the device flag (the step is then skipped) instead of the L1 / zero fallbacks,
    which only exist to keep the reference's loop alive."""
    base = _base_frame(reconstructed)
    loss, _ = ops.recon_mse(base if base is not None else reconstructed.contiguous(), original, flag)
    return loss


@torch.no_grad()
def calculate_anomaly_scores(model, test_loader, device="cuda"):
    """cad1:526-564: (0.7 * per-clip reconstruction error + 0.3 * memory score, labels, recon errors, memory scores)."""
    model.eval()
    dev = torch.device(device)
    scores, labels_all, recons, mems = [], [], [], []
    for videos, labels in test_loader:
        videos = videos.to(dev, non_blocking=True)
        out = model(videos)
        base = _base_frame(out["reconstructed"])
        _, clip = ops.recon_mse(base if base is not None else out["reconstructed"].contiguous(), videos)
        mem = out["anomaly_score"]
        scores.append(0.7 * clip + 0.3 * mem)
        recons.append(clip)
        mems.append(mem)
        labels_all.extend(np.asarray(labels).tolist())
    cat = lambda xs: torch.cat(xs).cpu().numpy() if xs else np.zeros(0, dtype=np.float32)   # noqa: E731
    return cat(scores), np.array(labels_all), cat(recons), cat(mems)


class MDTrainer:
    """Loop body of cad1:380-425: reconstruction loss, memory update, clip 0.1, Adam(lr, L2 decay 1e-6), skip on non-finite."""

    def __init__(self, model, device, lr=5e-7, dp=None):
        self.device = torch.device(device) if not isinstance(device, torch.device) else device
        if self.device.type != "cuda":
            raise RuntimeError("M-D trainer (cvad_b200) requires a CUDA device; there is no CPU fallback")
        self.model = model.to(self.device)
        self.optimizer = FusedAdam(list(self.model.parameters()), lr=lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-6, decoupled=False,
                                   clip_mode=1, max_norm=0.1, nan_mode=1)
        self.scheduler = torch.optim.lr_scheduler.ReduceLROnPlateau(self.optimizer, mode="min", factor=0.8, patience=3, min_lr=1e-7)
        if dp is not None:
            dp.attach(self.optimizer)

    def train_step(self, videos):
        self.optimizer.zero_grad()
        out = self.model(videos)
        loss = reconstruction_loss(videos, out["reconstructed"], self.optimizer.arena.header[0:1])
        self.model.update_memory(out["sequence_feature"])
        loss.backward()
        self.optimizer.step()
        return loss, out


def train_model(model, train_loader, val_loader, num_epochs=30, lr=5e-7, device="cuda", verbose=True):
    """cad1:346-524 without the plotting: returns (model, train_losses, val_losses)."""
    tr = MDTrainer(model, device, lr)
    train_losses, val_losses = [], []
    for epoch in range(num_epochs):
        tr.model.train()
        acc = torch.zeros(2, device=tr.device)
        for videos, _ in train_loader:
            loss, _ = tr.train_step(videos.to(tr.device, non_blocking=True))
            ok = torch.isfinite(loss).float()
            acc[0] += torch.nan_to_num(loss.detach()) * ok
            acc[1] += ok
        tr.model.eval()
        vacc = torch.zeros(2, device=tr.device)
        with torch.no_grad():
            for videos, _ in val_loader:
                videos = videos.to(tr.device, non_blocking=True)
                vacc[0] += reconstruction_loss(videos, tr.model(videos)["reconstructed"])
                vacc[1] += 1
        a, v = acc.tolist(), vacc.tolist()
        train_losses.append(a[0] / max(a[1], 1))
        val_losses.append(v[0] / max(v[1], 1))
        tr.scheduler.step(val_losses[-1])
        if verbose:
            print(f"Epoch {epoch + 1}/{num_epochs}, Train Loss: {train_losses[-1]:.6f}, Val Loss: {val_losses[-1]:.6f}")
    return tr.model, train_losses, val_losses
