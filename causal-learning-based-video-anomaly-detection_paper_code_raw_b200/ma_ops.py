"""autograd glue for the M-A causal-branch kernels (csrc/ma_tail.cu, csrc/ma_branch.cu; ABI in include/cvad_b200.h)."""
from __future__ import annotations

import torch

from .ops import _call, _cuda, _f32c, _ptr, _ptr_array, _st, grad_buffer, _wants_grad

MAXDET, NF, HID = 5, 6, 64


class _DetDecode(torch.autograd.Function):
    """raw (B,T,5,4) -> box (B,T,5,4); cnt (B,T) int32 and src (B,T,5) int32 are returned non-differentiable."""

    @staticmethod
    def forward(ctx, raw, flag):
        _cuda(raw)
        raw = _f32c(raw)
        B, T = raw.shape[:2]
        R = B * T
        box = torch.empty((B, T, MAXDET, 4), device=raw.device, dtype=torch.float32)
        cnt = torch.empty((B, T), device=raw.device, dtype=torch.int32)
        src = torch.empty((B, T, MAXDET), device=raw.device, dtype=torch.int32)
        _call("cvad_det_decode_f32", _ptr(raw), R, _ptr(box), _ptr(cnt), _ptr(src), _ptr(flag), _st())
        ctx.save_for_backward(raw, src)
        ctx.mark_non_differentiable(cnt, src)
        return box, cnt, src

    @staticmethod
    def backward(ctx, dbox, _c, _s):
        raw, src = ctx.saved_tensors
        dbox = _f32c(dbox)
        draw = torch.empty_like(raw)
        _call("cvad_det_decode_bwd_f32", _ptr(raw), _ptr(dbox), _ptr(src), src.numel() // MAXDET, _ptr(draw), _st())
        return draw, None


def det_decode(raw, flag=None):
    return _DetDecode.apply(raw, flag)


class _TrajAssemble(torch.autograd.Function):
    """box (B,T,5,4), reid (B,T,5,D), cnt (B,T) -> traj (B,5,T,4+D), ntr (B) int32."""

    @staticmethod
    def forward(ctx, box, reid, cnt, flag):
        _cuda(box, reid, cnt)
        box, reid = _f32c(box), _f32c(reid)
        B, T = box.shape[:2]
        D = reid.shape[-1]
        traj = torch.empty((B, MAXDET, T, 4 + D), device=box.device, dtype=torch.float32)
        ntr = torch.empty((B,), device=box.device, dtype=torch.int32)
        _call("cvad_traj_assemble_f32", _ptr(box), _ptr(reid), _ptr(cnt), B, T, D, _ptr(traj), _ptr(ntr), _ptr(flag), _st())
        ctx.save_for_backward(cnt)
        ctx.meta = (B, T, D)
        ctx.mark_non_differentiable(ntr)
        return traj, ntr

    @staticmethod
    def backward(ctx, dtraj, _n):
        (cnt,) = ctx.saved_tensors
        B, T, D = ctx.meta
        dtraj = _f32c(dtraj)
        dbox = torch.empty((B, T, MAXDET, 4), device=dtraj.device, dtype=torch.float32)
        dreid = torch.empty((B, T, MAXDET, D), device=dtraj.device, dtype=torch.float32)
        _call("cvad_traj_assemble_bwd_f32", _ptr(dtraj), _ptr(cnt), B, T, D, _ptr(dbox), _ptr(dreid), _st())
        return dbox, dreid, None, None


def traj_assemble(box, reid, cnt, flag=None):
    return _TrajAssemble.apply(box, reid, cnt, flag)


class _GruLast(torch.autograd.Function):
    """gi (B*5,T,192) precomputed input projection -> last hidden state (B*5,64)."""

    @staticmethod
    def forward(ctx, gi, w_hh, b_hh, ntr):
        _cuda(gi, w_hh, b_hh, ntr)
        gi = _f32c(gi)
        N, T, _ = gi.shape
        B = N // MAXDET
        hT = torch.empty((N, HID), device=gi.device, dtype=torch.float32)
        need = any(ctx.needs_input_grad)
        saved = torch.empty((N, T, 5, HID), device=gi.device, dtype=torch.float32) if need else None
        _call("cvad_gru_fwd_f32", _ptr(gi), _ptr(w_hh), _ptr(b_hh), _ptr(ntr), B, T, _ptr(hT), _ptr(saved), _st())
        ctx.save_for_backward(saved, ntr)
        ctx.w_hh, ctx.b_hh = w_hh, b_hh
        ctx.meta = (B, T)
        return hT

    @staticmethod
    def backward(ctx, dhT):
        saved, ntr = ctx.saved_tensors
        B, T = ctx.meta
        w_hh, b_hh = ctx.w_hh, ctx.b_hh
        dhT = _f32c(dhT)
        dgi = torch.empty((B * MAXDET, T, 3 * HID), device=dhT.device, dtype=torch.float32)
        dw = grad_buffer(w_hh) if _wants_grad(w_hh) else None
        db = grad_buffer(b_hh) if _wants_grad(b_hh) else None
        _call("cvad_gru_bwd_f32", _ptr(dhT), _ptr(saved), _ptr(w_hh), _ptr(ntr), B, T, _ptr(dgi), _ptr(dw), _ptr(db), _st())
        return dgi, None, None, None


def gru_last(gi, w_hh, b_hh, ntr):
    return _GruLast.apply(gi, w_hh, b_hh, ntr)


class _ReparamKl(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mu, lv, eps, ntr):
        _cuda(mu, lv, eps, ntr)
        mu, lv, eps = _f32c(mu), _f32c(lv), _f32c(eps)
        B = ntr.shape[0]
        z = torch.empty((B, MAXDET, NF), device=mu.device, dtype=torch.float32)
        kl = torch.empty((B,), device=mu.device, dtype=torch.float32)
        _call("cvad_reparam_kl_f32", _ptr(mu), _ptr(lv), _ptr(eps), _ptr(ntr), B, _ptr(z), _ptr(kl), _st())
        ctx.save_for_backward(mu, lv, eps, ntr)
        return z, kl

    @staticmethod
    def backward(ctx, dz, dkl):
        mu, lv, eps, ntr = ctx.saved_tensors
        B = ntr.shape[0]
        dz, dkl = _f32c(dz), _f32c(dkl)
        dmu, dlv = torch.empty_like(mu), torch.empty_like(lv)
        _call("cvad_reparam_kl_bwd_f32", _ptr(mu), _ptr(lv), _ptr(eps), _ptr(ntr), B, _ptr(dz), _ptr(dkl), _ptr(dmu), _ptr(dlv), _st())
        return dmu, dlv, None, None


def reparam_kl(mu, lv, eps, ntr):
    return _ReparamKl.apply(mu, lv, eps, ntr)


class _PairConcat(torch.autograd.Function):
    @staticmethod
    def forward(ctx, node):
        _cuda(node)
        node = _f32c(node)
        B, _, Hn = node.shape
        pair = torch.empty((B, MAXDET, MAXDET, 2 * Hn), device=node.device, dtype=torch.float32)
        _call("cvad_pair_concat_f32", _ptr(node), B, Hn, _ptr(pair), _st())
        ctx.meta = (B, Hn)
        return pair

    @staticmethod
    def backward(ctx, dpair):
        B, Hn = ctx.meta
        dpair = _f32c(dpair)
        dnode = torch.empty((B, MAXDET, Hn), device=dpair.device, dtype=torch.float32)
        _call("cvad_pair_concat_bwd_f32", _ptr(dpair), B, Hn, _ptr(dnode), _st())
        return dnode


def pair_concat(node):
    return _PairConcat.apply(node)


class _AdjAssemble(torch.autograd.Function):
    @staticmethod
    def forward(ctx, e, ntr):
        _cuda(e, ntr)
        e = _f32c(e)
        B = ntr.shape[0]
        adj = torch.empty((B, NF, NF), device=e.device, dtype=torch.float32)
        _call("cvad_adj_assemble_f32", _ptr(e), _ptr(ntr), B, _ptr(adj), 0, _st())
        ctx.save_for_backward(ntr)
        ctx.eshape = e.shape
        return adj

    @staticmethod
    def backward(ctx, dadj):
        (ntr,) = ctx.saved_tensors
        B = ntr.shape[0]
        dadj = _f32c(dadj)
        de = torch.empty(ctx.eshape, device=dadj.device, dtype=torch.float32)
        _call("cvad_adj_assemble_f32", _ptr(dadj), _ptr(ntr), B, _ptr(de), 1, _st())
        return de, None


def adj_assemble(e, ntr):
    return _AdjAssemble.apply(e, ntr)


class _Structured(torch.autograd.Function):
    @staticmethod
    def forward(ctx, adj, z):
        _cuda(adj, z)
        adj, z = _f32c(adj), _f32c(z)
        B = adj.shape[0]
        out = torch.empty_like(z)
        _call("cvad_structured_f32", _ptr(adj), _ptr(z), B, _ptr(out), _st())
        ctx.save_for_backward(adj, z)
        return out

    @staticmethod
    def backward(ctx, dout):
        adj, z = ctx.saved_tensors
        dout = _f32c(dout)
        dadj, dz = torch.empty_like(adj), torch.empty_like(z)
        _call("cvad_structured_bwd_f32", _ptr(adj), _ptr(z), _ptr(dout), adj.shape[0], _ptr(dadj), _ptr(dz), _st())
        return dadj, dz


def structured(adj, z):
    return _Structured.apply(adj, z)


# (in, out) of the 20 nn.Linear layers of the causal branch, in the order of cvad_ma_branch_*_f32's params (include/cvad_b200.h)
BRANCH_LAYERS = ((64, 32), (32, 32), (32, 32), (32, 6), (32, 6), (6, 32), (64, 32), (32, 1), (6, 32), (32, 32), (32, 6), (18, 64), (64, 32),
                 (32, 1), (12, 32), (32, 16), (16, 1), (6, 32), (32, 16), (16, 1))


class _CausalBranch(torch.autograd.Function):
    """hT (B*5,64), ntr (B) int32, eps (B,5,6), keep (B,64) or None, 40 parameters -> z (B,5,6), kl (B), adj (B,6,6), causal (B).
    Parameter gradients are added into ``grad_buffer(p)`` on the current stream; the backward recomputes the forward."""

    @staticmethod
    def forward(ctx, hT, ntr, eps, keep, *params):
        _cuda(hT, ntr, eps, keep, *params)
        for i, p in enumerate(params):
            din, dout = BRANCH_LAYERS[i // 2]
            if tuple(p.shape) != ((dout, din) if i % 2 == 0 else (dout,)) or p.dtype != torch.float32 or not p.is_contiguous():
                raise ValueError(f"causal_branch: parameter {i} has shape {tuple(p.shape)} / {p.dtype}; the kernel is built for the "
                                 "reference's layer widths (num_factors = 6) in contiguous fp32")
        hT, eps = _f32c(hT), _f32c(eps)
        keep = None if keep is None else _f32c(keep)
        ntr = ntr.to(torch.int32).contiguous()
        B = ntr.shape[0]
        dev = hT.device
        z = torch.empty((B, MAXDET, NF), device=dev, dtype=torch.float32)
        kl = torch.empty((B,), device=dev, dtype=torch.float32)
        adj = torch.empty((B, NF, NF), device=dev, dtype=torch.float32)
        causal = torch.empty((B,), device=dev, dtype=torch.float32)
        _call("cvad_ma_branch_fwd_f32", _ptr(hT), _ptr(ntr), _ptr(eps), _ptr(keep), B, _ptr_array(params), _ptr(z), _ptr(kl), _ptr(adj),
              _ptr(causal), _st())
        ctx.save_for_backward(hT, ntr, eps, keep)
        ctx.params = params
        ctx.set_materialize_grads(False)      # an output without a gradient reaches the kernel as NULL, not as a tensor of zeros
        return z, kl, adj, causal

    @staticmethod
    def backward(ctx, dz, dkl, dadj, dcausal):
        hT, ntr, eps, keep = ctx.saved_tensors
        params = ctx.params
        dz, dkl, dadj, dcausal = (None if g is None else _f32c(g) for g in (dz, dkl, dadj, dcausal))
        dhT = torch.empty_like(hT)
        grads = [grad_buffer(p) if _wants_grad(p) else None for p in params]
        _call("cvad_ma_branch_bwd_f32", _ptr(hT), _ptr(ntr), _ptr(eps), _ptr(keep), ntr.shape[0], _ptr_array(params), _ptr(dz), _ptr(dkl),
              _ptr(dadj), _ptr(dcausal), _ptr(dhT), _ptr_array(grads), _st())
        return (dhT if ctx.needs_input_grad[0] else None, None, None, None) + (None,) * len(params)


def causal_branch(hT, ntr, eps, keep, params):
    """M-A's causal branch behind the GRU (cad:300-502) as one kernel forward and one backward.  ``params``: the 40 weight / bias tensors
    in the order of BRANCH_LAYERS; ``keep``: the causal scorer's dropout keep-mask (training) or None."""
    return _CausalBranch.apply(hT, ntr, eps, keep, *params)


class _SoftmaxRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        _cuda(x)
        x = _f32c(x)
        y = torch.empty_like(x)
        _call("cvad_softmax_rows_f32", _ptr(x), x.numel() // x.shape[-1], x.shape[-1], _ptr(y), _st())
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        dy = _f32c(dy)
        dx = torch.empty_like(y)
        _call("cvad_softmax_rows_bwd_f32", _ptr(y), _ptr(dy), y.numel() // y.shape[-1], y.shape[-1], _ptr(dx), _st())
        return dx


def softmax_rows(x):
    return _SoftmaxRows.apply(x)
