"""Deterministic synthetic inputs / weights shared by tools/make_golden.py, the tests, smoke() and bench.py.

Everything is drawn from ``torch.Generator`` on the CPU with explicit seeds so the golden
generator (which runs next to /root/reference) and the GPU-box tests (which cannot see it)
rebuild bit-identical tensors without shipping them.  SURVEY.md section 8(d) defines the shapes.
"""
from __future__ import annotations

import math
import os

import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# A checkpoint with AdamW state is stored in three files so that none exceeds 1 MB: ``<name>`` without the two moment tensors of each
# optimizer state entry, and ``<stem>.exp_avg.pt`` / ``<stem>.exp_avg_sq.pt`` holding them as lists in state order.
MOMENTS = ("exp_avg", "exp_avg_sq")


def _moment_paths(name):
    stem = name.rsplit(".", 1)[0]
    return {m: os.path.join(GOLDEN, f"{stem}.{m}.pt") for m in MOMENTS}


def golden(name):
    """The committed fixture ``tests/golden/<name>``; a split checkpoint comes back whole."""
    d = torch.load(os.path.join(GOLDEN, name), map_location="cpu", weights_only=False)
    parts = _moment_paths(name)
    if all(os.path.exists(p) for p in parts.values()):
        moments = {m: torch.load(p, map_location="cpu", weights_only=True) for m, p in parts.items()}
        for i, st in enumerate(d["optimizer_state_dict"]["state"].values()):
            st.update((m, moments[m][i]) for m in MOMENTS)
    return d


def save_golden_checkpoint(ck, name):
    """Store a checkpoint with AdamW state as ``golden(name)`` reads it back."""
    opt = ck["optimizer_state_dict"]
    state = {i: {k: v for k, v in st.items() if k not in MOMENTS} for i, st in opt["state"].items()}
    torch.save({**ck, "optimizer_state_dict": {**opt, "state": state}}, os.path.join(GOLDEN, name))
    for m, p in _moment_paths(name).items():
        torch.save([st[m] for st in opt["state"].values()], p)


def gen(seed: int) -> torch.Generator:
    return torch.Generator().manual_seed(int(seed))


def mb_clips(B, T, H=64, W=64, seed=1234):
    """M-B / s1 / s2 input: rand(B,3,T,H,W) in [0,1) (C3 of SURVEY 8d, brightness factor optional)."""
    return torch.rand(B, 3, T, H, W, generator=gen(seed))


def mb_clips_bright(B, T, H=64, W=64, seed=1234):
    g = gen(seed)
    x = torch.rand(B, 3, T, H, W, generator=g)
    return x * torch.rand(B, 1, 1, 1, 1, generator=g)


def mc_clips(B, T, H=64, W=64, seed=1234):
    """M-C input: rand(B,1,T,H,W) in [0,1) (mc3:118-122 semantics)."""
    return torch.rand(B, 1, T, H, W, generator=gen(seed))


def ma_clips(B, T, H=240, W=360, seed=1234, wide=True):
    """M-A input (B,T,1,H,W).  wide=True reproduces cad:96,1177-1179: raw 0..255 floats through
    Normalize(0.5,0.5) => [-1, 509]; wide=False gives the [-1,1] variant."""
    g = gen(seed)
    if wide:
        x = torch.randint(0, 256, (B, T, 1, H, W), generator=g).float()
        return (x - 0.5) / 0.5
    return torch.rand(B, T, 1, H, W, generator=g) * 2 - 1


def md_clips(B, T, H=64, W=64, seed=1234):
    """M-D input (B,T,1,H,W) in [0.001, 0.999] (cad1:110-114 semantics)."""
    return torch.rand(B, T, 1, H, W, generator=gen(seed)) * 0.998 + 0.001


def keep_mask(shape, p, seed):
    """Dropout keep-mask (1 = keep) with drop probability p."""
    return (torch.rand(*shape, generator=gen(seed)) >= p).float()


def synth_fill(state: dict, seed: int, skip=()) -> dict:
    """Overwrite every floating tensor of a state_dict (in key order) with reproducible values
    scaled like torch's default init; BN statistics get trained-like non-trivial values."""
    out = {}
    for i, (k, v) in enumerate(state.items()):
        if any(s in k for s in skip) or not torch.is_floating_point(v):
            out[k] = v.clone()
            continue
        g = gen(seed * 1000 + i)
        if k.endswith("running_var"):
            t = torch.rand(v.shape, generator=g) + 0.5
        elif k.endswith("running_mean"):
            t = (torch.rand(v.shape, generator=g) - 0.5) * 0.4
        elif v.dim() == 1 and (".bn" in k or _is_bn_key(k, state)):
            t = torch.rand(v.shape, generator=g) + 0.5 if k.endswith("weight") else (torch.rand(v.shape, generator=g) - 0.5) * 0.4
        else:
            fan_in = v[0].numel() if v.dim() > 1 else max(v.numel(), 1)
            bound = 1.0 / math.sqrt(max(fan_in, 1))
            if v.dim() == 1:
                # bias: bound from the matching weight's fan-in when present
                wk = k[: -len("bias")] + "weight" if k.endswith("bias") else None
                if wk in state and state[wk].dim() > 1:
                    bound = 1.0 / math.sqrt(state[wk][0].numel())
            t = (torch.rand(v.shape, generator=g) * 2 - 1) * bound
        out[k] = t.to(v.dtype)
    return out


def _is_bn_key(k: str, state: dict) -> bool:
    base = k.rsplit(".", 1)[0]
    return (base + ".running_mean") in state


def summarize(t: torch.Tensor, n: int = 16) -> dict:
    """Compact fingerprint of a tensor for golden comparison of large gradients."""
    f = t.detach().double().flatten()
    return {"norm": float(f.norm()), "sum": float(f.sum()), "absmax": float(f.abs().max()) if f.numel() else 0.0,
            "head": t.detach().flatten()[:n].clone(), "numel": t.numel()}


def is_bn_fed_conv_bias(key: str) -> bool:
    """M-A backbone convolution biases (layerX.0.bias / layerX.3.bias): BatchNorm subtracts the batch mean right after them, so their
    gradient is analytically zero; the reference accumulates pure round-off there (and Adam amplifies it to +-lr steps)."""
    parts = key.split(".")
    return len(parts) == 4 and parts[0] == "backbone" and parts[1].startswith("layer") and parts[2] in ("0", "3") and parts[3] == "bias"


def strided_sample(t: torch.Tensor, cap: int = 16384) -> torch.Tensor:
    """Every k-th element of a tensor (k chosen so that at most ``cap`` remain): a compact stand-in for large parameter tensors."""
    f = t.detach().flatten()
    k = max(1, (f.numel() + cap - 1) // cap)
    return f[::k].clone()
