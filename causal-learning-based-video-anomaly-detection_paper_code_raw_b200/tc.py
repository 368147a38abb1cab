"""bf16 tensor-core execution of the M-A backbone (cad:141-158): one autograd node for the whole conv/BN/ReLU stack.

Data flow per step.  Activations live in HBM as zero-bordered NHWC bf16 ("padded-flat", (N, H+2, W+2, C)); the input of a
stride-2 convolution is written by its producer as four phase planes instead (see csrc/flatconv_tc.cu), so every one of
the eight 3x3 convolutions -- forward, data-gradient and weight-gradient -- is a sum of row-shifted GEMMs that TMA feeds
straight into tcgen05.mma.  Statistics and parameter gradients are fp32.

  x fp32 (B*T,1,240,360) --2x2 space-to-depth--> X4 (16-byte pixels) --tcgen05 tf32 conv, pass 1: bn1 batch statistics
      --pass 2: conv + BN + ReLU--> bf16 NHWC --MaxPool(3,2,1)--> a0 bf16 padded-flat (.,62,92,32)
  for the 8 layers: raw_i = flatconv(a_{i-1}) ; (mean, invstd) = stats(raw_i) ; a_i = relu(bn(raw_i)) [plain | phase planes]
  features = AdaptiveAvgPool(4,6)(a_8) -> fp32 (B*T, 6144) in the reference's (c,h,w) order

Backward walks the same list in reverse: ReLU+BN backward, tcgen05 weight-gradient (fp32 atomics into the gradient arena) and
tcgen05 data-gradient.  The BatchNorm backward of every training-mode layer below the top one is one pass over raw and dact: its two
per-channel sums come from the convolution above -- sum g from the data-gradient's epilogue under the ReLU bitmask the forward apply
wrote, sum act*dact = sum W*dW from the staged weight gradient (include/cvad_b200.h, cvad_pad_bn_relu_bwd_tsum_bf16).  The top layer
(its dact comes from the average pool) and the configurations without a staged main-stream weight gradient take a reduce pass first.  Convolution biases that feed a BatchNorm have an analytically zero
gradient (the reference only accumulates round-off there); they receive exactly zero here.
"""
from __future__ import annotations

import contextlib
import os

import torch

from . import ops
from .ops import _call, _ptr, _st, grad_buffer, _wants_grad

BF16 = torch.bfloat16
STAGED_WGRAD = os.environ.get("CVAD_STAGED_WGRAD", "1") != "0"      # weight-gradient atomics through a [tap][Cout][Cin] staging buffer
_WG_SCRATCH = {}


def _wgrad_scratch(device, cin, cout):
    """Zeroed staging buffer of a layer shape (stream-ordered reuse: every call leaves it zero again)."""
    key = (str(device), int(cin), int(cout))
    buf = _WG_SCRATCH.get(key)
    if buf is None:
        buf = _WG_SCRATCH[key] = torch.zeros(9 * cin * cout, device=device, dtype=torch.float32)
    return buf


STEM_FUSED_POOL = os.environ.get("CVAD_STEM_FUSED_POOL", "1") != "0"   # stem pass 2 + max-pool as one kernel
STEM_F16 = os.environ.get("CVAD_STEM_F16", "1") != "0"                 # fp16 stem over a 2x4 space-to-depth (frame width % 4 == 0)
FUSED_STATS = os.environ.get("CVAD_FUSED_BN_STATS", "1") != "0"     # BatchNorm batch statistics from the convolution epilogue
# weight-gradient GEMMs on a side stream: wgrad_i needs only draw_i and a_{i-1}, so it can run beside the HBM-bound BatchNorm backward of
# the next layer down instead of in front of it (a parallel branch of the captured step graph)
WGRAD_OVERLAP = os.environ.get("CVAD_WGRAD_OVERLAP", "0") == "1"


def _layers(bb):
    out = []
    for layer in (bb.layer1, bb.layer2, bb.layer3, bb.layer4):
        for ci, bi in ((0, 1), (3, 4)):
            out.append((layer[ci], layer[bi]))
    return out


def out_hw(h, w, stride):
    return (h - 1) // stride + 1, (w - 1) // stride + 1


def act_shape(N, h, w, c, phase):
    """Buffer shape of an activation with interior (h, w): padded-flat, or the 4 phase planes of the stride-2 conv reading it."""
    if not phase:
        return (N, h + 2, w + 2, c)
    ho, wo = out_hw(h, w, 2)
    return (4, N, ho + 2, wo + 2, c)


class _BackboneBF16(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, bb, *params):
        dev = x.device
        N, _, H, W = x.shape
        st = _st()
        # ---- stem (frozen in the reference's training recipe, cad:596-598): tf32 tensor-core conv, two passes over x
        bn1, conv1 = bb.bn1, bb.conv1
        C1 = conv1.out_channels
        if C1 != 32 or conv1.in_channels != 1 or conv1.kernel_size != (7, 7) or conv1.stride != (2, 2):
            raise RuntimeError("the tensor-core stem implements the reference's 7x7 stride-2 1->32 convolution (cad:115)")
        x = x.contiguous()
        need_bwd = any(ctx.needs_input_grad)
        layers = _layers(bb)
        strides = [conv.stride[0] for conv, _ in layers]
        if strides[0] == 2:
            raise RuntimeError("the first 3x3 convolution after the stem is stride 1 in the reference (cad:150)")
        # bf16 weight packs of the eight 3x3 layers: independent of the activations, so they are issued on a side stream beside the
        # stem and joined before the first 3x3 convolution (allocated here, on the compute stream, which also consumes them)
        packs, cin = [], C1
        for i, (conv, _) in enumerate(layers):
            cout = conv.out_channels
            wf = torch.empty((9 * cout, cin), device=dev, dtype=BF16)
            wd = torch.empty((9 * cin, cout), device=dev, dtype=BF16) if need_bwd and i > 0 else None
            packs.append((wf, wd))
            cin = cout
        cur, side = torch.cuda.current_stream(), ops.aux_stream(dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            cin = C1
            for (conv, _), (wf, wd), stride in zip(layers, packs, strides):
                _call("cvad_flat_pack_w3x3_bf16", _ptr(conv.weight), conv.out_channels, cin, stride, _ptr(wf), _ptr(wd), _st())
                cin = conv.out_channels
        H1, W1 = out_hw(H, W, 2)
        mean = torch.empty(C1, device=dev, dtype=torch.float32)
        invstd = torch.empty_like(mean)
        w1, b1 = conv1.weight.detach(), conv1.bias.detach()
        h, w = out_hw(H1, W1, 2)
        a = torch.empty(act_shape(N, h, w, C1, False), device=dev, dtype=BF16)

        def bn1_statistics(entry, xs):
            if bn1.training:
                _call(entry, _ptr(xs), _ptr(w1), _ptr(b1), N, H, W, _ptr(ops.bn_workspace(dev, C1)), float(bn1.eps), float(bn1.momentum),
                      _ptr(mean), _ptr(invstd), _ptr(bn1.running_mean), _ptr(bn1.running_var), _ptr(bn1.num_batches_tracked), st)
            else:
                _call("cvad_bn_eval_prepare_f32", C1, float(bn1.eps), _ptr(bn1.running_mean), _ptr(bn1.running_var), _ptr(mean), _ptr(invstd), st)

        stem_forward(bb, x, a, mean, invstd, bn1_statistics)
        del x
        cur.wait_stream(side)
        saved = []
        cin = C1
        # ReLU bitmask of layer i for its (S1, T) backward: a training-mode BatchNorm under a convolution whose weight gradient runs staged
        # on this stream (T is read from its staging buffer, and it must be complete before layer i's backward)
        ts_ok = need_bwd and STAGED_WGRAD and not WGRAD_OVERLAP
        for i, (conv, bn) in enumerate(layers):
            cout, stride = conv.out_channels, strides[i]
            wf, wd = packs[i]
            ho, wo = out_hw(h, w, stride)
            raw = torch.empty((N, ho + 2, wo + 2, cout), device=dev, dtype=BF16)
            mean = torch.empty(cout, device=dev, dtype=torch.float32)
            invstd = torch.empty_like(mean)
            fused = bn.training and FUSED_STATS and cout in (32, 64, 128, 256)
            if fused:
                # batch statistics straight from the convolution's epilogue (no second pass over raw); the finalize rides in the apply pass
                ws = ops.bn_workspace(dev, cout)
                _call("cvad_flat_conv3x3_fwd_stats_bf16", _ptr(a), _ptr(wf), _ptr(conv.bias), _ptr(raw), N, h, w, cin, cout, stride, _ptr(ws), st)
            elif bn.training:
                _call("cvad_flat_conv3x3_fwd_bf16", _ptr(a), _ptr(wf), _ptr(conv.bias), _ptr(raw), N, h, w, cin, cout, stride, st)
                _call("cvad_pad_bn_stats_bf16", _ptr(raw), N, ho, wo, cout, _ptr(ops.bn_workspace(dev, cout)), float(bn.eps), float(bn.momentum),
                      _ptr(mean), _ptr(invstd), _ptr(bn.running_mean), _ptr(bn.running_var), _ptr(bn.num_batches_tracked), st)
            else:
                _call("cvad_flat_conv3x3_fwd_bf16", _ptr(a), _ptr(wf), _ptr(conv.bias), _ptr(raw), N, h, w, cin, cout, stride, st)
                _call("cvad_bn_eval_prepare_f32", cout, float(bn.eps), _ptr(bn.running_mean), _ptr(bn.running_var), _ptr(mean), _ptr(invstd), st)
            phase_out = i + 1 < len(layers) and strides[i + 1] == 2
            act = torch.empty(act_shape(N, ho, wo, cout, phase_out), device=dev, dtype=BF16)
            mask = None
            if ts_ok and bn.training and i + 1 < len(layers) and _wants_grad(layers[i + 1][0].weight):
                mask = torch.empty(act.numel() // 8, device=dev, dtype=torch.uint8)
            if fused:
                _call("cvad_pad_bn_finalize_apply_relu_mask_bf16" if mask is not None else "cvad_pad_bn_finalize_apply_relu_bf16", _ptr(raw),
                      _ptr(act), *((_ptr(mask),) if mask is not None else ()), N, ho, wo, cout, int(phase_out), _ptr(ws), float(bn.eps),
                      float(bn.momentum), _ptr(bn.weight), _ptr(bn.bias), _ptr(mean), _ptr(invstd), _ptr(bn.running_mean), _ptr(bn.running_var),
                      _ptr(bn.num_batches_tracked), st)
            else:
                _call("cvad_pad_bn_apply_relu_mask_bf16" if mask is not None else "cvad_pad_bn_apply_relu_bf16", _ptr(raw), _ptr(act),
                      *((_ptr(mask),) if mask is not None else ()), N, ho, wo, cout, int(phase_out), _ptr(mean), _ptr(invstd), _ptr(bn.weight),
                      _ptr(bn.bias), st)
            if need_bwd:
                saved.append((a, raw, mean, invstd, wd, (h, w, cin, cout, stride, ho, wo), bn.training, phase_out, mask))
            a, h, w, cin = act, ho, wo, cout
        feats = torch.empty((N, cin, 4, 6), device=dev, dtype=torch.float32)
        _call("cvad_pad_avgpool_bf16_fwd", _ptr(a), N, h, w, cin, 4, 6, _ptr(feats), st)
        ctx.bb, ctx.saved, ctx.last = bb, saved, (N, h, w, cin)
        return feats.reshape(N, -1)

    @staticmethod
    def backward(ctx, dfeat):
        bb, saved = ctx.bb, ctx.saved
        if any(sv is None for sv in saved):
            raise RuntimeError("cvad_b200 bf16 backbone: backward called a second time; the saved activations are released layer by layer "
                               "during the first backward (retain_graph is not supported on this path)")
        N, h, w, c = ctx.last
        st = _st()
        dev = dfeat.device
        dfeat = ops._f32c(dfeat)
        dact = torch.empty((N, h + 2, w + 2, c), device=dev, dtype=BF16)
        _call("cvad_pad_avgpool_bf16_bwd", _ptr(dfeat), N, h, w, c, 4, 6, _ptr(dact), st)
        layers = _layers(bb)
        cur = torch.cuda.current_stream()
        side = ops.aux_stream(dev, 1) if WGRAD_OVERLAP else None
        keep = []                     # operands of side-stream launches stay referenced until the join (the allocator tracks one stream)
        for idx in range(len(layers) - 1, -1, -1):
            conv, bn = layers[idx]
            a_in, raw, mean, invstd, wd, (hi, wi, cin, cout, stride, ho, wo), bn_training, phase_out, mask = saved[idx]
            draw = torch.empty_like(raw)
            dg = grad_buffer(bn.weight) if _wants_grad(bn.weight) else None
            db = grad_buffer(bn.bias) if _wants_grad(bn.bias) else None
            if mask is not None:    # sum g and sum act*dact are already in the workspace (taken by the convolution above)
                _call("cvad_pad_bn_relu_bwd_tsum_bf16", _ptr(raw), _ptr(dact), _ptr(draw), N, ho, wo, cout, int(phase_out), _ptr(mean), _ptr(invstd),
                      _ptr(bn.weight), _ptr(bn.bias), _ptr(ops.bn_workspace(dev, cout)), _ptr(dg), _ptr(db), st)
            else:
                _call("cvad_pad_bn_relu_bwd_bf16", _ptr(raw), _ptr(dact), _ptr(draw), N, ho, wo, cout, int(phase_out), _ptr(mean), _ptr(invstd),
                      _ptr(bn.weight), _ptr(bn.bias), int(bn_training), _ptr(ops.bn_workspace(dev, cout)), _ptr(dg), _ptr(db), st)
            mask_lo = saved[idx - 1][8] if idx > 0 else None      # the layer below takes its sums from this layer's convolution
            if _wants_grad(conv.weight):
                wst = st
                if side is not None:
                    side.wait_stream(cur)
                    keep.append((a_in, draw))
                    wst = side.cuda_stream
                with torch.cuda.stream(side) if side is not None else contextlib.nullcontext():
                    if mask_lo is not None:
                        _call("cvad_flat_conv3x3_wgrad_staged_wdot_bf16", _ptr(a_in), _ptr(draw), _ptr(grad_buffer(conv.weight)),
                              _ptr(_wgrad_scratch(dev, cin, cout)), N, hi, wi, cin, cout, stride, _ptr(conv.weight), _ptr(ops.bn_workspace(dev, cin)),
                              wst)
                    elif STAGED_WGRAD:
                        _call("cvad_flat_conv3x3_wgrad_staged_bf16", _ptr(a_in), _ptr(draw), _ptr(grad_buffer(conv.weight)),
                              _ptr(_wgrad_scratch(dev, cin, cout)), N, hi, wi, cin, cout, stride, wst)
                    else:
                        _call("cvad_flat_conv3x3_wgrad_bf16", _ptr(a_in), _ptr(draw), _ptr(grad_buffer(conv.weight)), N, hi, wi, cin, cout, stride, wst)
            if _wants_grad(conv.bias):
                grad_buffer(conv.bias)          # analytically zero (BatchNorm removes the mean); keep the tensor "with grad"
            if idx > 0:
                dact = torch.empty(a_in.shape, device=dev, dtype=BF16)
                if mask_lo is not None:
                    # dact is the gradient w.r.t. relu(bn(raw_lo)): its epilogue also takes sum g under the ReLU mask of that layer
                    _call("cvad_flat_conv3x3_dgrad_masksum_bf16", _ptr(draw), _ptr(wd), _ptr(dact), N, hi, wi, cin, cout, stride, _ptr(mask_lo),
                          _ptr(ops.bn_workspace(dev, cin)), st)
                else:
                    _call("cvad_flat_conv3x3_dgrad_bf16", _ptr(draw), _ptr(wd), _ptr(dact), N, hi, wi, cin, cout, stride, st)
            saved[idx] = None
        if side is not None:
            cur.wait_stream(side)
            keep.clear()
        return (None, None) + (None,) * (len(ctx.needs_input_grad) - 2)


def stem_forward(bb, x, a, mean, invstd, bn1_statistics=None):
    """The stem conv1 -> bn1 -> ReLU -> MaxPool(3,2,1) of x (N,1,H,W) (uint8 raw frames or normalised fp32, contiguous) into ``a``, the
    padded-flat (N, h+2, w+2, 32) bf16 input of layer1.  Takes the fp16 stem over a 2x4 space-to-depth when the frame width allows it,
    else the tf32 stem with pass 2 fused with the pool, else the unfused tf32 stem and a separate pool.  ``bn1_statistics(entry, xs)``
    fills (mean, invstd) between the space-to-depth and pass 2 (``entry``: the batch-statistics entry point of the chosen stem over
    its space-to-depth ``xs``); None: they already hold bn1's."""
    N, _, H, W = x.shape
    dev, st = x.device, _st()
    bn1, conv1 = bb.bn1, bb.conv1
    C1 = conv1.out_channels
    H1, W1 = out_hw(H, W, 2)
    w1, b1 = conv1.weight.detach(), conv1.bias.detach()
    n8 = int(ops.L().cvad_stem8_bytes(N, H, W)) if (STEM_F16 and STEM_FUSED_POOL) else -1
    if n8 >= 0:
        # fp16 stem over a 2x4 space-to-depth (frame width a multiple of 4): 6 MMAs of N = 64 per 256 outputs, pass 2 fused with the pool
        x8 = torch.empty(n8, device=dev, dtype=torch.uint8)
        if x.dtype == torch.uint8:  # raw frames: Normalize(mean, std) of cad:1177-1179 applied on the fly
            _call("cvad_stem8_space_to_depth_u8", _ptr(x), N, H, W, float(bb.input_mean), float(bb.input_std), _ptr(x8), st)
        else:
            _call("cvad_stem8_space_to_depth_f32", _ptr(x), N, H, W, _ptr(x8), st)
        if bn1_statistics is not None:
            bn1_statistics("cvad_stem8_f16_stats", x8)
        _call("cvad_stem8_f16_bn_relu_maxpool", _ptr(x8), _ptr(w1), _ptr(b1), N, H, W, _ptr(mean), _ptr(invstd), _ptr(bn1.weight),
              _ptr(bn1.bias), _ptr(a), st)
        return
    n4 = int(ops.L().cvad_stem_x4_floats(N, H, W))
    if n4 < 0:
        raise RuntimeError(f"frame size {H}x{W} is outside the tensor-core stem's range")
    x4 = torch.empty(n4, device=dev, dtype=torch.float32)       # 2x2 space-to-depth of the batch: 16-byte pixels
    if x.dtype == torch.uint8:
        _call("cvad_stem_space_to_depth_u8", _ptr(x), N, H, W, float(bb.input_mean), float(bb.input_std), _ptr(x4), st)
    else:
        _call("cvad_stem_space_to_depth_f32", _ptr(x), N, H, W, _ptr(x4), st)
    if bn1_statistics is not None:
        bn1_statistics("cvad_stem_tf32_stats", x4)
    fused = 801
    if STEM_FUSED_POOL:
        # pass 2 and MaxPool(3,2,1) in one kernel: the 708 MB tensor between them stays in shared memory (801 = a band does not fit)
        fused = _call("cvad_stem_tf32_bn_relu_maxpool", _ptr(x4), _ptr(w1), _ptr(b1), N, H, W, _ptr(mean), _ptr(invstd), _ptr(bn1.weight),
                      _ptr(bn1.bias), _ptr(a), st, accept=(801,))
    if fused == 801:
        y1 = torch.empty((N, H1, W1, C1), device=dev, dtype=BF16)
        _call("cvad_stem_tf32_bn_relu", _ptr(x4), _ptr(w1), _ptr(b1), N, H, W, _ptr(mean), _ptr(invstd), _ptr(bn1.weight), _ptr(bn1.bias),
              _ptr(y1), st)
        _call("cvad_pad_maxpool3x3s2_bf16", _ptr(y1), N, H1, W1, C1, _ptr(a), st)


def backbone_forward_bf16(bb, x):
    """x (B*T, 1, H, W) fp32 -> features (B*T, 6144) fp32."""
    ops._cuda(x)
    if torch.is_grad_enabled() and any(p.requires_grad for p in list(bb.conv1.parameters()) + list(bb.bn1.parameters())):
        # the backward stops at layer1.0: no gradient is computed for the stem.  That is the reference's training recipe
        # (apply_memory_efficient_training freezes backbone.conv1 / backbone.bn1, cad:596-598); anything else must not train silently
        # with all-zero stem gradients
        raise RuntimeError("cvad_b200 bf16 backbone: backbone.conv1 / backbone.bn1 require grad, but the tensor-core path has no stem "
                           "backward; freeze them (apply_memory_efficient_training, cad:596-598) or use set_precision('fp32')")
    params = [p for p in bb.parameters() if p.requires_grad]
    x = x.contiguous() if x.dtype == torch.uint8 else x.float().contiguous()
    return _BackboneBF16.apply(x, bb, *params)


# ---- layout helpers (host side; used by the tests and by callers that want NCHW views of the flat buffers)
def to_padded(x_nchw):
    """(N,C,H,W) -> padded-flat (N,H+2,W+2,C) bf16 with a zero border."""
    N, C, H, W = x_nchw.shape
    out = torch.zeros((N, H + 2, W + 2, C), device=x_nchw.device, dtype=BF16)
    out[:, 1:H + 1, 1:W + 1, :] = x_nchw.permute(0, 2, 3, 1).to(BF16)
    return out


def from_padded(buf, H, W):
    return buf[:, 1:H + 1, 1:W + 1, :].permute(0, 3, 1, 2).float().contiguous()


def to_phase(x_nchw):
    """(N,C,H,W) -> the four phase planes (4,N,Ho+2,Wo+2,C) a stride-2 flat convolution reads."""
    N, C, H, W = x_nchw.shape
    ho, wo = out_hw(H, W, 2)
    xp = torch.zeros((N, 2 * (ho + 2) + 2, 2 * (wo + 2) + 2, C), device=x_nchw.device, dtype=BF16)
    xp[:, 3:H + 3, 3:W + 3, :] = x_nchw.permute(0, 2, 3, 1).to(BF16)      # xp[r] = padded(r - 2)
    planes = [xp[:, a:a + 2 * (ho + 2):2, b:b + 2 * (wo + 2):2, :] for a in (0, 1) for b in (0, 1)]
    return torch.stack(planes, 0).contiguous()


def from_phase(planes, H, W):
    """Inverse of to_phase for the interior pixels: (4,N,Ho+2,Wo+2,C) -> (N,C,H,W) fp32."""
    _, N, hq, wq, C = planes.shape
    full = torch.zeros((N, 2 * hq, 2 * wq, C), device=planes.device, dtype=planes.dtype)
    k = 0
    for a in (0, 1):
        for b in (0, 1):
            full[:, a::2, b::2, :] = planes[k]
            k += 1
    return full[:, 3:H + 3, 3:W + 3, :].permute(0, 3, 1, 2).float().contiguous()
