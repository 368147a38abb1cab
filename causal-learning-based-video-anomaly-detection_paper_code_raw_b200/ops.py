"""torch.autograd glue over the C ABI (include/cvad_b200.h).  PyTorch owns memory, streams and the autograd graph;
every FLOP on the hot path runs in the hand-written sm_100a kernels of libcvad_b200.so.  No CPU path exists: CPU
tensors raise.

Gradient convention: parameter gradients are ACCUMULATED IN PLACE into ``param.grad`` by the weight-gradient kernels
(``param.grad`` is normally a view into the flat gradient arena of ``arena.FlatArena`` so that the gradient all-reduce
and the fused optimizer see one contiguous buffer); the autograd Functions return ``None`` for parameters.
"""
from __future__ import annotations

import contextlib
import ctypes
import os

import torch

from . import _lib
from ._lib import ConvDesc, check

ACT_NONE, ACT_RELU, ACT_LEAKY01, ACT_SIGMOID, ACT_TANH = 0, 1, 2, 3, 4

LAUNCHES = [0]   # number of cvad kernels-launching ABI calls issued (bench.py reports it as gpu_launches evidence)


def L():
    return _lib.lib()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("cvad_b200 ops run only on CUDA tensors (sm_100a); there is no CPU fallback")


def _ptr(t):
    return None if t is None else t.data_ptr()


TIMED = {}        # bench.py: ABI name -> list of (start_event, end_event); set TIMED_NAMES to enable
TIMED_NAMES = set()
TIMED_CAPTURE_ONLY = [False]     # True: bracket the named calls only while a CUDA graph is being captured
TIMED_SHAPES = [os.environ.get("CVAD_PROFILE_SHAPES", "0") == "1"]


def _call(name, *args, accept=()):
    """Invoke one C-ABI entry point; raises on a non-zero status unless it is listed in ``accept`` (then it is returned: e.g. 801 =
    "this fused variant does not fit, use the unfused calls")."""
    LAUNCHES[0] += 1
    timed = (name in TIMED_NAMES or "*" in TIMED_NAMES) and (not TIMED_CAPTURE_ONLY[0] or torch.cuda.is_current_stream_capturing())
    if timed:
        # inside a capture the events become event-record nodes of the graph ("external" events): every replay re-records
        # them, so elapsed_time() measures the call as it runs inside the replayed step
        ext = torch.cuda.is_current_stream_capturing()
        s = torch.cuda.Event(enable_timing=True, external=ext)
        e = torch.cuda.Event(enable_timing=True, external=ext)
        s.record()
    status = getattr(L(), name)(*args)
    if status in accept and status != 0:
        LAUNCHES[0] -= 1
        return status
    check(status, name)
    if timed:
        e.record()
        key = name
        if TIMED_SHAPES[0] and name == "cvad_sgemm_f32":        # profiling detail: one row per GEMM shape
            key = f"{name}[M{args[0]} N{args[1]} K{args[2]} splits{args[16]}{' gated' if args[17] else ''}]"
        TIMED.setdefault(key, []).append((s, e))
    return 0


class _ParamGradOverlap:
    """Side stream for the parameter-gradient kernels of the dense layers (weight-gradient GEMM, bias column sums).

    In a backward pass only the data-gradient chain is on the critical path; the ~70 small weight/bias-gradient launches of the
    M-A tail merely have to finish before the optimizer (or the gradient all-reduce) reads the arena.  Inside
    ``param_grad_overlap()`` they are issued on a second stream that forks from the current stream at every layer and joins when the
    context exits; in a captured step the fork/join become graph edges, so the two chains run concurrently on replay.  Their
    operands are kept alive until the join (the caching allocator only tracks the stream a block was allocated on)."""
    active = False
    streams = {}
    keep = []


_AUX_STREAMS = {}


def aux_stream(device, which: int = 0):
    """Extra streams per device for work that is independent of the critical chain (callers fork and join explicitly)."""
    st = _AUX_STREAMS.get((device.index, which))
    if st is None:
        st = _AUX_STREAMS[(device.index, which)] = torch.cuda.Stream(device=device)
    return st


def _pg_stream(device):
    if not _ParamGradOverlap.active:
        return None
    st = _ParamGradOverlap.streams.get(device.index)
    if st is None:
        st = _ParamGradOverlap.streams[device.index] = torch.cuda.Stream(device=device)
    return st


@contextlib.contextmanager
def param_grad_overlap(enabled: bool = True):
    if not enabled or os.environ.get("CVAD_PG_OVERLAP", "1") == "0" or _ParamGradOverlap.active:
        yield
        return
    _ParamGradOverlap.active = True
    try:
        yield
    finally:
        _ParamGradOverlap.active = False
        if _ParamGradOverlap.keep:
            cur = torch.cuda.current_stream()
            for st in _ParamGradOverlap.streams.values():
                if st.device == cur.device:
                    cur.wait_stream(st)
            _ParamGradOverlap.keep.clear()


def grad_buffer(p: torch.Tensor) -> torch.Tensor:
    """The fp32 buffer wgrad kernels accumulate into (the arena view when the parameter is arena-managed)."""
    if p.grad is None:
        p.grad = torch.zeros_like(p, memory_format=torch.contiguous_format)
    return p.grad


def _wants_grad(p) -> bool:
    return p is not None and p.requires_grad


def _f32c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def zeros_f32(shape, device):
    """fp32 zeros through the library's own fill kernel (the accumulating GEMMs / reductions need zeroed outputs every step)."""
    t = torch.empty(shape, device=device, dtype=torch.float32)
    if t.numel():
        _call("cvad_fill_f32", _ptr(t), t.numel(), 0.0, _st())
    return t


def u8_normalize(x: torch.Tensor, mean: float, std: float) -> torch.Tensor:
    """uint8 frames -> fp32 ``(x - mean) / std`` (torchvision Normalize on the reference's FloatTensor frames, cad:1177-1179)."""
    _cuda(x)
    x = x.contiguous()
    y = torch.empty(x.shape, device=x.device, dtype=torch.float32)
    _call("cvad_u8_normalize_f32", _ptr(x), x.numel(), float(mean), float(std), _ptr(y), _st())
    return y


# ------------------------------------------------------------------------------------------------ convolution
def _conv_desc(x5, w5, y5, stride, padding) -> ConvDesc:
    d = ConvDesc()
    d.N, d.Cin, d.Din, d.Hin, d.Win = x5.shape
    d.Cout, d.Dout, d.Hout, d.Wout = y5.shape[1:]
    d.kD, d.kH, d.kW = w5.shape[2:]
    d.sD, d.sH, d.sW = stride
    d.pD, d.pH, d.pW = padding
    for i in range(5):
        d.xs[i] = x5.stride(i)
        d.ys[i] = y5.stride(i)
    return d


def _triple(v, nd):
    if isinstance(v, int):
        v = (v,) * nd
    v = tuple(v)
    return (1,) * (3 - nd) + v if nd < 3 else v


def _pad3(v, nd):
    if isinstance(v, int):
        v = (v,) * nd
    v = tuple(v)
    return (0,) * (3 - nd) + v if nd < 3 else v


class _ConvAct(torch.autograd.Function):
    """act(conv(x, w) + b) for 2-D (N,C,H,W) or 3-D (N,C,D,H,W) inputs."""

    @staticmethod
    def forward(ctx, x, weight, bias, stride, padding, act):
        _cuda(x, weight, bias)
        nd = x.dim() - 2
        x = x if x.dtype == torch.float32 else x.float()
        x5 = x if nd == 3 else x.unsqueeze(2)
        w5 = weight if nd == 3 else weight.unsqueeze(2)
        s3, p3 = _triple(stride, nd), _pad3(padding, nd)
        N, _, Di, Hi, Wi = x5.shape
        Co, _, kD, kH, kW = w5.shape
        Do = (Di + 2 * p3[0] - kD) // s3[0] + 1
        Ho = (Hi + 2 * p3[1] - kH) // s3[1] + 1
        Wo = (Wi + 2 * p3[2] - kW) // s3[2] + 1
        y5 = torch.empty((N, Co, Do, Ho, Wo), device=x.device, dtype=torch.float32)
        d = _conv_desc(x5, w5, y5, s3, p3)
        _call("cvad_conv_fwd_f32", ctypes.byref(d), _ptr(x5), _ptr(weight), _ptr(bias), _ptr(y5), act, _st())
        ctx.geom = (s3, p3, act, nd)
        ctx.weight, ctx.bias = weight, bias
        ctx.save_for_backward(x5, y5 if act != ACT_NONE else None)
        return y5 if nd == 3 else y5.squeeze(2)

    @staticmethod
    def backward(ctx, dy):
        x5, y5 = ctx.saved_tensors
        s3, p3, act, nd = ctx.geom
        weight, bias = ctx.weight, ctx.bias
        dy5 = _f32c(dy if nd == 3 else dy.unsqueeze(2))
        if act != ACT_NONE:
            dz = torch.empty_like(dy5)
            _call("cvad_act_mask_bwd_f32", _ptr(dy5), _ptr(y5), None, 1.0, act, _ptr(dz), dy5.numel(), _st())
            dy5 = dz
        w5 = weight if nd == 3 else weight.unsqueeze(2)
        d = _conv_desc(x5, w5, dy5, s3, p3)
        if _wants_grad(weight):
            _call("cvad_conv_wgrad_f32", ctypes.byref(d), _ptr(x5), _ptr(dy5), _ptr(grad_buffer(weight)), _st())
        if _wants_grad(bias):
            N, Co = dy5.shape[:2]
            _call("cvad_channel_sum_add_f32", _ptr(dy5), N, Co, dy5[0, 0].numel(), _ptr(grad_buffer(bias)), _st())
        dx = None
        if ctx.needs_input_grad[0]:
            dx5 = torch.empty(x5.shape, device=x5.device, dtype=torch.float32)
            dd = _conv_desc(dx5, w5, dy5, s3, p3)
            _call("cvad_conv_dgrad_f32", ctypes.byref(dd), _ptr(dy5), _ptr(weight), _ptr(dx5), 0, _st())
            dx = dx5 if nd == 3 else dx5.squeeze(2)
        return dx, None, None, None, None, None


def conv_act(x, weight, bias, stride=1, padding=0, act=ACT_NONE):
    return _ConvAct.apply(x, weight, bias, stride, padding, act)


def bn_fold_conv(weight, bias, bn):
    """(w', b') of the convolution that equals conv followed by ``bn`` in eval mode (running statistics)."""
    _cuda(weight)
    w = _f32c(weight.detach())
    wf = torch.empty_like(w)
    bf = torch.empty(w.shape[0], device=w.device, dtype=torch.float32)
    _call("cvad_bn_fold_conv_f32", _ptr(w), _ptr(bias), _ptr(bn.weight), _ptr(bn.bias), _ptr(bn.running_mean), _ptr(bn.running_var), float(bn.eps),
          w.shape[0], w[0].numel(), _ptr(wf), _ptr(bf), _st())
    return wf, bf


# ------------------------------------------------------------------------------------------------ linear
def _sgemm(M, N, K, A, lda, a_k, B, ldb, b_k, C, ldc, bias=None, act=ACT_NONE, mask=None, mask_scale=1.0, accumulate=0, splits=1, gate=None):
    _call("cvad_sgemm_f32", M, N, K, _ptr(A), lda, int(a_k), _ptr(B), ldb, int(b_k), _ptr(C), ldc, _ptr(bias), act, _ptr(mask),
          float(mask_scale), int(accumulate), int(splits), _ptr(gate), _st())


TF32X3 = os.environ.get("CVAD_TF32X3", "1") != "0"      # tensor-core (3xTF32) forward of the wide projections


def _splits_for(M, N, K):
    """Split the reduction over gridDim.z whenever the 64x64 output tiles alone cannot fill the 148 SMs."""
    tiles = ((M + 63) // 64) * ((N + 63) // 64)
    if tiles >= 148 or K < 128:
        return 1
    return max(1, min(K // 64, (2 * 148) // tiles))


class _LinearAct(torch.autograd.Function):
    """act(x @ W^T + b) * keep_mask / (1-p) over the last axis of x.  ``gate``: optional device scalar; when it is 0 at
    backward time the layer's gradient GEMMs are skipped on the device and dx is exactly zero."""

    @staticmethod
    def forward(ctx, x, weight, bias, act, mask, mask_scale, gate):
        _cuda(x, weight, bias, mask)
        shp = x.shape
        x2 = _f32c(x).reshape(-1, shp[-1])
        M, K = x2.shape
        O = weight.shape[0]
        splits = _splits_for(M, O, K)
        if mask is not None:
            mask = _f32c(mask).reshape(M, O)
        if TF32X3 and K >= 2048 and K % 32 == 0 and O >= 128 and x2.data_ptr() % 16 == 0 and weight.data_ptr() % 16 == 0:
            # the two 6144 -> 512 projections: tcgen05 kind::tf32 with the 3xTF32 split (fp32-level accuracy), split-K + atomic reduction
            y = zeros_f32((M, O), x.device)
            _call("cvad_linear_fwd_tf32x3", _ptr(x2), _ptr(weight), _ptr(y), M, O, K, _st())
            if bias is not None or act != ACT_NONE or mask is not None:
                _call("cvad_bias_act_mask_f32", _ptr(y), M, O, _ptr(bias), act, _ptr(mask), float(mask_scale), _st())
        elif splits > 1:
            y = zeros_f32((M, O), x.device)
            _sgemm(M, O, K, x2, K, True, weight, K, True, y, O, splits=splits)
            if bias is not None or act != ACT_NONE or mask is not None:
                _call("cvad_bias_act_mask_f32", _ptr(y), M, O, _ptr(bias), act, _ptr(mask), float(mask_scale), _st())
        else:
            y = torch.empty((M, O), device=x.device, dtype=torch.float32)
            _sgemm(M, O, K, x2, K, True, weight, K, True, y, O, bias, act, mask, mask_scale)
        ctx.meta = (act, mask_scale, shp)
        ctx.weight, ctx.bias, ctx.gate = weight, bias, gate
        ctx.save_for_backward(x2, y if act != ACT_NONE else None, mask)
        return y.reshape(*shp[:-1], O)

    @staticmethod
    def backward(ctx, dy):
        x2, y, mask = ctx.saved_tensors
        act, mask_scale, shp = ctx.meta
        weight, bias, gate = ctx.weight, ctx.bias, ctx.gate
        M, K = x2.shape
        O = weight.shape[0]
        dz = _f32c(dy).reshape(M, O)
        if act != ACT_NONE or mask is not None:
            out = torch.empty_like(dz)
            _call("cvad_act_mask_bwd_f32", _ptr(dz), _ptr(y), _ptr(mask), float(mask_scale), act, _ptr(out), dz.numel(), _st())
            dz = out
        gw = grad_buffer(weight) if _wants_grad(weight) else None
        gb = grad_buffer(bias) if _wants_grad(bias) else None
        side = _pg_stream(dz.device) if (gw is not None or gb is not None) else None
        if side is not None:         # off the critical path: fork here, join when param_grad_overlap() exits
            side.wait_stream(torch.cuda.current_stream())
            _ParamGradOverlap.keep.append((dz, x2))
        with (torch.cuda.stream(side) if side is not None else contextlib.nullcontext()):
            if gw is not None:       # dW[o][i] += sum_m dz[m][o] x[m][i]
                _sgemm(O, K, M, dz, O, False, x2, K, False, gw, K, accumulate=1, splits=_splits_for(O, K, M), gate=gate)
            if gb is not None:
                _call("cvad_colsum_f32", _ptr(dz), M, O, O, _ptr(gb), 1, _st())
        dx = None
        if ctx.needs_input_grad[0]:  # dx[m][i] = sum_o dz[m][o] W[o][i]
            splits = _splits_for(M, K, O)
            if splits > 1 or gate is not None:
                dx = zeros_f32((M, K), dz.device)
            else:
                dx = torch.empty((M, K), device=dz.device, dtype=torch.float32)
            _sgemm(M, K, O, dz, O, True, weight, K, False, dx, K, splits=splits, gate=gate)
            dx = dx.reshape(shp)
        return dx, None, None, None, None, None, None


def linear_act(x, weight, bias, act=ACT_NONE, mask=None, p_drop=0.0, gate=None):
    scale = 1.0 / (1.0 - p_drop) if mask is not None else 1.0
    return _LinearAct.apply(x, weight, bias, act, mask, scale, gate)



# ------------------------------------------------------------------------------------------------ fused MLP chains
CHAIN_MAX_DIM, CHAIN_MAX_LAYERS, CHAIN_MAX_W = 256, 8, 50000
FUSED_CHAINS = os.environ.get("CVAD_FUSED_CHAINS", "1") != "0"


def _ptr_array(items):
    arr = (ctypes.c_void_p * len(items))()
    for i, t in enumerate(items):
        arr[i] = None if t is None else t.data_ptr()
    return arr


class _MLPChain(torch.autograd.Function):
    """A stack of nn.Linear layers (width <= 512) with activation / dropout keep-masks as one launch forward and one launch for the
    data-gradient chain; weight and bias gradients are the usual split-K GEMMs / column sums on the parameter-gradient side stream."""

    @staticmethod
    def forward(ctx, x, acts, scales, n, *tensors):
        weights, biases, masks = tensors[:n], tensors[n:2 * n], tensors[2 * n:3 * n]
        _cuda(x, *weights)
        shp = x.shape
        x2 = _f32c(x).reshape(-1, shp[-1])
        M = x2.shape[0]
        dims = [x2.shape[1]] + [w.shape[0] for w in weights]
        masks = [None if m is None else _f32c(m).reshape(M, d) for m, d in zip(masks, dims[1:])]
        need = torch.is_grad_enabled() or any(ctx.needs_input_grad)
        saves = [torch.empty((M, d), device=x.device, dtype=torch.float32) if need else None for d in dims[1:]]
        out = saves[-1] if need else torch.empty((M, dims[-1]), device=x.device, dtype=torch.float32)
        c_dims, c_acts = (ctypes.c_int * (n + 1))(*dims), (ctypes.c_int * n)(*acts)
        c_scales = (ctypes.c_float * n)(*scales)
        # the last layer's stored output IS the result: the kernel writes it through `saves` and `out` (same buffer)
        _call("cvad_mlp_chain_fwd_f32", _ptr(x2), M, n, c_dims, c_acts, _ptr_array(weights), _ptr_array(biases), _ptr_array(masks), c_scales,
              _ptr_array(saves), _ptr(out), _st())
        ctx.meta = (acts, scales, n, shp, dims)
        ctx.params = (weights, biases)
        ctx.save_for_backward(x2, *[s for s in saves if s is not None], *[m for m in masks if m is not None])
        ctx.mask_slots = [m is not None for m in masks]
        return out.reshape(*shp[:-1], dims[-1])

    @staticmethod
    def backward(ctx, dy):
        acts, scales, n, shp, dims = ctx.meta
        weights, biases = ctx.params
        sv = ctx.saved_tensors
        x2, saves = sv[0], list(sv[1:1 + n])
        it = iter(sv[1 + n:])
        masks = [next(it) if has else None for has in ctx.mask_slots]
        M = x2.shape[0]
        dy2 = _f32c(dy).reshape(M, dims[-1])
        dzs = [torch.empty((M, d), device=dy2.device, dtype=torch.float32) for d in dims[1:]]
        dx = torch.empty((M, dims[0]), device=dy2.device, dtype=torch.float32) if ctx.needs_input_grad[0] else None
        c_dims, c_acts = (ctypes.c_int * (n + 1))(*dims), (ctypes.c_int * n)(*acts)
        c_scales = (ctypes.c_float * n)(*scales)
        _call("cvad_mlp_chain_bwd_f32", _ptr(dy2), M, n, c_dims, c_acts, _ptr_array(weights), _ptr_array(masks), c_scales, _ptr_array(saves),
              _ptr_array(dzs), _ptr(dx), _st())
        side = _pg_stream(dy2.device)
        if side is not None:         # off the critical path: fork here, join when param_grad_overlap() exits
            side.wait_stream(torch.cuda.current_stream())
            _ParamGradOverlap.keep.append((dzs, x2, saves))
        with (torch.cuda.stream(side) if side is not None else contextlib.nullcontext()):
            for l in range(n):
                w, b, dz = weights[l], biases[l], dzs[l]
                hin = x2 if l == 0 else saves[l - 1]
                O, K = dims[l + 1], dims[l]
                if _wants_grad(w):       # dW[o][i] += sum_m dz[m][o] h[m][i]
                    _sgemm(O, K, M, dz, O, False, hin, K, False, grad_buffer(w), K, accumulate=1, splits=_splits_for(O, K, M))
                if _wants_grad(b):
                    _call("cvad_colsum_f32", _ptr(dz), M, O, O, _ptr(grad_buffer(b)), 1, _st())
        return (None if dx is None else dx.reshape(shp), None, None, None) + (None,) * (3 * n)


def mlp_chain(x, layers):
    """``layers``: sequence of (weight, bias, act, keep_mask or None, p_drop).  Equivalent to chaining ``linear_act`` over them."""
    n = len(layers)
    assert 1 <= n <= CHAIN_MAX_LAYERS
    acts = tuple(int(l[2]) for l in layers)
    scales = tuple((1.0 / (1.0 - l[4])) if l[3] is not None else 1.0 for l in layers)
    return _MLPChain.apply(x, acts, scales, n, *[l[0] for l in layers], *[l[1] for l in layers], *[l[3] for l in layers])


def chainable(layers, din) -> bool:
    """Whether a Linear stack fits the fused kernel: widths <= 256 and all weight matrices together small enough for shared memory."""
    if not FUSED_CHAINS or not 1 <= len(layers) <= CHAIN_MAX_LAYERS or din > CHAIN_MAX_DIM:
        return False
    if any(l[0].shape[0] > CHAIN_MAX_DIM for l in layers):
        return False
    return sum(((l[0].shape[1] | 1) * l[0].shape[0] + 3) // 4 * 4 for l in layers) <= CHAIN_MAX_W


# ------------------------------------------------------------------------------------------------ batch norm
class _BatchNormAct(torch.autograd.Function):
    """BatchNorm + activation applied to ``groups`` consecutive slices of the batch axis as separate calls, in order: what the
    reference does when it runs the frame encoder once per time step (cad1:227-231): per-step batch statistics and ``groups``
    sequential running-statistics updates.  groups = 1 is the ordinary op."""

    @staticmethod
    def forward(ctx, x, gamma, beta, running_mean, running_var, nbt, ws, training, act, eps, momentum, groups):
        _cuda(x, gamma, beta)
        x = _f32c(x)
        NT, C = x.shape[:2]
        assert NT % groups == 0
        N = NT // groups
        S = x[0, 0].numel()
        mean = torch.empty((groups, C), device=x.device, dtype=torch.float32)
        invstd = torch.empty_like(mean)
        y = torch.empty_like(x)
        for gi in range(groups):
            xs, ys = x[gi * N:(gi + 1) * N], y[gi * N:(gi + 1) * N]
            if training:
                _call("cvad_bn_train_stats_f32", _ptr(xs), N, C, S, _ptr(ws), float(eps), float(momentum), _ptr(mean[gi]), _ptr(invstd[gi]),
                      _ptr(running_mean), _ptr(running_var), _ptr(nbt), _st())
            else:
                _call("cvad_bn_eval_prepare_f32", C, float(eps), _ptr(running_mean), _ptr(running_var), _ptr(mean[gi]), _ptr(invstd[gi]), _st())
            _call("cvad_bn_apply_f32", _ptr(xs), _ptr(ys), N, C, S, _ptr(mean[gi]), _ptr(invstd[gi]), _ptr(gamma), _ptr(beta), act, _st())
        ctx.meta = (training, act, groups)
        ctx.gamma, ctx.beta, ctx.ws = gamma, beta, ws
        ctx.save_for_backward(x, mean, invstd)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, mean, invstd = ctx.saved_tensors
        training, act, groups = ctx.meta
        gamma, beta, ws = ctx.gamma, ctx.beta, ctx.ws
        dy = _f32c(dy)
        NT, C = x.shape[:2]
        N = NT // groups
        S = x[0, 0].numel()
        dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        dg = grad_buffer(gamma) if _wants_grad(gamma) else None
        db = grad_buffer(beta) if _wants_grad(beta) else None
        if dx is None and dg is None and db is None:
            return (None,) * 12
        for gi in range(groups):
            sl = slice(gi * N, (gi + 1) * N)
            _call("cvad_bn_bwd_f32", _ptr(dy[sl]), _ptr(x[sl]), _ptr(dx[sl]) if dx is not None else None, N, C, S, _ptr(mean[gi]),
                  _ptr(invstd[gi]), _ptr(gamma), _ptr(beta), act, int(training), _ptr(ws), _ptr(dg), _ptr(db), _st())
        return (dx,) + (None,) * 11


def batchnorm_act(x, gamma, beta, running_mean, running_var, nbt, ws, training, act=ACT_NONE, eps=1e-5, momentum=0.1, groups=1):
    return _BatchNormAct.apply(x, gamma, beta, running_mean, running_var, nbt, ws, training, act, eps, momentum, groups)


# ------------------------------------------------------------------------------------------------ pooling
class _MaxPool(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, kernel, stride, padding):
        _cuda(x)
        nd = x.dim() - 2
        x = _f32c(x)
        k3, s3, p3 = _triple(kernel, nd), _triple(stride, nd), _pad3(padding, nd)
        x5 = x if nd == 3 else x.unsqueeze(2)
        N, C, D, H, W = x5.shape
        OD = (D + 2 * p3[0] - k3[0]) // s3[0] + 1
        OH = (H + 2 * p3[1] - k3[1]) // s3[1] + 1
        OW = (W + 2 * p3[2] - k3[2]) // s3[2] + 1
        y = torch.empty((N, C, OD, OH, OW), device=x.device, dtype=torch.float32)
        need_idx = ctx.needs_input_grad[0]
        idx = torch.empty((N, C, OD, OH, OW), device=x.device, dtype=torch.int32) if need_idx else None
        _call("cvad_maxpool_fwd_f32", _ptr(x5), _ptr(y), _ptr(idx), N * C, D, H, W, OD, OH, OW, *k3, *s3, *p3, _st())
        ctx.meta = (x5.shape, nd)
        ctx.save_for_backward(idx)
        return y if nd == 3 else y.squeeze(2)

    @staticmethod
    def backward(ctx, dy):
        (idx,) = ctx.saved_tensors
        shape5, nd = ctx.meta
        dy = _f32c(dy)
        N, C, D, H, W = shape5
        dx = torch.zeros(shape5, device=dy.device, dtype=torch.float32)
        _call("cvad_maxpool_bwd_f32", _ptr(dy), _ptr(idx), _ptr(dx), N * C, D * H * W, idx[0, 0].numel(), _st())
        return (dx if nd == 3 else dx.squeeze(2)), None, None, None


def maxpool(x, kernel, stride=None, padding=0):
    return _MaxPool.apply(x, kernel, stride if stride is not None else kernel, padding)


class _AdaptiveAvgPool(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, out_size):
        _cuda(x)
        nd = x.dim() - 2
        x = _f32c(x)
        x5 = x if nd == 3 else x.unsqueeze(2)
        o3 = _triple(out_size, nd)
        N, C, D, H, W = x5.shape
        y = torch.empty((N, C) + tuple(o3), device=x.device, dtype=torch.float32)
        _call("cvad_adaptive_avgpool_fwd_f32", _ptr(x5), _ptr(y), N * C, D, H, W, *o3, _st())
        ctx.meta = (x5.shape, o3, nd)
        return y if nd == 3 else y.squeeze(2)

    @staticmethod
    def backward(ctx, dy):
        shape5, o3, nd = ctx.meta
        dy = _f32c(dy)
        N, C, D, H, W = shape5
        dx = torch.empty(shape5, device=dy.device, dtype=torch.float32)
        _call("cvad_adaptive_avgpool_bwd_f32", _ptr(dy), _ptr(dx), N * C, D, H, W, *o3, _st())
        return (dx if nd == 3 else dx.squeeze(2)), None


def adaptive_avgpool(x, out_size):
    return _AdaptiveAvgPool.apply(x, out_size)


class _MeanMid(torch.autograd.Function):
    """(A,T,F) -> (A,F) mean over T."""

    @staticmethod
    def forward(ctx, x):
        _cuda(x)
        x = _f32c(x)
        A, T, F = x.shape
        y = torch.empty((A, F), device=x.device, dtype=torch.float32)
        _call("cvad_mean_mid_fwd_f32", _ptr(x), _ptr(y), A, T, F, _st())
        ctx.meta = (A, T, F)
        return y

    @staticmethod
    def backward(ctx, dy):
        A, T, F = ctx.meta
        dy = _f32c(dy)
        dx = torch.empty((A, T, F), device=dy.device, dtype=torch.float32)
        _call("cvad_mean_mid_bwd_f32", _ptr(dy), _ptr(dx), A, T, F, 0, _st())
        return dx


def mean_mid(x):
    return _MeanMid.apply(x)


# ------------------------------------------------------------------------------------------------ losses
class _MbLoss(torch.autograd.Function):
    """s2:135-205.  Returns (total, components[8]); gradients w.r.t. scores and adj come from the same kernel pass."""

    @staticmethod
    def forward(ctx, scores, adj, pseudo, weights, flag):
        _cuda(scores, adj, pseudo)
        B = adj.shape[0]
        s = _f32c(scores).reshape(B)
        a = _f32c(adj).reshape(B, 256)
        ps = _f32c(pseudo).reshape(B)
        ws = torch.empty(int(L().cvad_mb_loss_ws_floats(B)), device=a.device, dtype=torch.float32)
        out = torch.empty(8, device=a.device, dtype=torch.float32)
        ds = torch.empty(B, device=a.device, dtype=torch.float32)
        da = torch.empty((B, 256), device=a.device, dtype=torch.float32)
        _call("cvad_mb_loss_f32", _ptr(s), _ptr(a), _ptr(ps), B, *[float(w) for w in weights], _ptr(ws), _ptr(out), _ptr(ds), _ptr(da),
              _ptr(flag), _st())
        ctx.save_for_backward(ds, da)
        ctx.shapes = (scores.shape, adj.shape)
        ctx.mark_non_differentiable(out)
        return out[0].clone(), out

    @staticmethod
    def backward(ctx, g_total, _g_out):
        ds, da = ctx.saved_tensors
        ss, sa = ctx.shapes
        # g_total is 1 for loss.backward(); scaling by a device scalar keeps general callers correct
        return (ds * g_total).reshape(ss), (da * g_total).reshape(sa), None, None, None


def mb_loss(scores, adj, pseudo, weights=(1.0, 0.01, 0.001, 0.01), flag=None):
    return _MbLoss.apply(scores, adj, pseudo, tuple(weights), flag)


class _BceLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, scores, targets, flag):
        _cuda(scores, targets)
        s = _f32c(scores).reshape(-1)
        y = _f32c(targets).reshape(-1)
        out = torch.empty(1, device=s.device, dtype=torch.float32)
        ds = torch.empty_like(s)
        _call("cvad_bce_loss_f32", _ptr(s), _ptr(y), s.numel(), _ptr(out), _ptr(ds), _ptr(flag), _st())
        ctx.save_for_backward(ds)
        ctx.shape = scores.shape
        return out[0]

    @staticmethod
    def backward(ctx, g):
        (ds,) = ctx.saved_tensors
        return (ds * g).reshape(ctx.shape), None, None


def bce_loss(scores, targets, flag=None):
    return _BceLoss.apply(scores, targets, flag)


class _MaLoss(torch.autograd.Function):
    """cad:649-662 on (direct_predictions (B,2), anomaly_scores (B,), causal_anomaly_scores (B,), kl (B,), labels (B,))."""

    @staticmethod
    def forward(ctx, probs, final, causal, kl, labels, flag):
        _cuda(probs, final, causal, kl, labels)
        B = probs.shape[0]
        p, f, c, k = _f32c(probs), _f32c(final), _f32c(causal), _f32c(kl)
        lab = labels.to(torch.int64).contiguous()
        out = torch.empty(5, device=p.device, dtype=torch.float32)
        dp, df, dc, dk = torch.empty_like(p), torch.empty_like(f), torch.empty_like(c), torch.empty_like(k)
        _call("cvad_ma_loss_f32", _ptr(p), _ptr(f), _ptr(c), _ptr(k), _ptr(lab), B, _ptr(out), _ptr(dp), _ptr(df), _ptr(dc), _ptr(dk),
              _ptr(flag), _st())
        ctx.save_for_backward(dp, df, dc, dk)
        ctx.mark_non_differentiable(out)
        return out[0].clone(), out

    @staticmethod
    def backward(ctx, g, _g2):
        dp, df, dc, dk = ctx.saved_tensors
        return dp * g, df * g, dc * g, dk * g, None, None


def ma_loss(probs, final, causal, kl, labels, flag=None):
    return _MaLoss.apply(probs, final, causal, kl, labels, flag)


class _LinComb2(torch.autograd.Function):
    """out = a*x + b*y[:, col]  (cad:574)."""

    @staticmethod
    def forward(ctx, x, a, y, col, b):
        _cuda(x, y)
        x = _f32c(x)
        y = _f32c(y)
        n = x.numel()
        out = torch.empty_like(x)
        ys = y.shape[1] if y.dim() == 2 else 1
        yv = y[:, col] if y.dim() == 2 else y
        _call("cvad_lincomb2_f32", _ptr(out), _ptr(x), 1, float(a), yv.data_ptr(), ys, float(b), n, _st())
        ctx.meta = (a, b, col, y.shape)
        return out

    @staticmethod
    def backward(ctx, g):
        a, b, col, yshape = ctx.meta
        g = _f32c(g)
        dx = torch.empty_like(g)
        _call("cvad_lincomb2_f32", _ptr(dx), _ptr(g), 1, float(a), _ptr(g), 1, 0.0, g.numel(), _st())
        dy = zeros_f32(yshape, g.device)
        tgt = dy[:, col] if len(yshape) == 2 else dy
        tmp = torch.empty_like(g)
        _call("cvad_lincomb2_f32", _ptr(tmp), _ptr(g), 1, float(b), _ptr(g), 1, 0.0, g.numel(), _st())
        tgt.copy_(tmp)
        return dx, None, dy, None, None


def lincomb2(x, a, y, col, b):
    return _LinComb2.apply(x, a, y, col, b)


# ------------------------------------------------------------------------------------------------ dropout / helpers
class _MaskScale(torch.autograd.Function):
    """y = x * keep_mask / (1-p): a Dropout that is not preceded by one of our GEMMs (mc3:61)."""

    @staticmethod
    def forward(ctx, x, mask, scale):
        _cuda(x, mask)
        y = _f32c(x).clone()
        mask = _f32c(mask)
        rows = y.numel() // y.shape[-1]
        _call("cvad_bias_act_mask_f32", _ptr(y), rows, y.shape[-1], None, ACT_NONE, _ptr(mask), float(scale), _st())
        ctx.save_for_backward(mask)
        ctx.scale = scale
        return y

    @staticmethod
    def backward(ctx, dy):
        (mask,) = ctx.saved_tensors
        dy = _f32c(dy)
        dx = torch.empty_like(dy)
        _call("cvad_act_mask_bwd_f32", _ptr(dy), None, _ptr(mask), float(ctx.scale), ACT_NONE, _ptr(dx), dy.numel(), _st())
        return dx, None, None


def mask_scale(x, mask, p_drop):
    return _MaskScale.apply(x, mask, 1.0 / (1.0 - p_drop))


_BN_WS = {}


def bn_workspace(device, C):
    """2*C zeroed fp64 accumulators shared by all BN layers of that width on a device (calls are stream-ordered and each
    call re-zeroes the buffer before returning)."""
    key = (str(device), int(C))
    ws = _BN_WS.get(key)
    if ws is None:
        ws = torch.zeros(2 * C, device=device, dtype=torch.float64)
        _BN_WS[key] = ws
    return ws


# ------------------------------------------------------------------------------------------------ M-D building blocks
class _ConvTranspose2d(torch.autograd.Function):
    """nn.ConvTranspose2d without bias (cad1:162-177).  Its forward IS the data-gradient kernel of the convolution that maps
    (Cout_T -> Cin_T) with the same weight tensor (Cin_T, Cout_T, kH, kW); its backward is that convolution's forward (dx)
    and weight-gradient (dw) with the roles of x and dy exchanged."""

    @staticmethod
    def forward(ctx, x, weight, stride, padding):
        _cuda(x, weight)
        x = _f32c(x)
        N, Ci, Hi, Wi = x.shape
        _, Co, kH, kW = weight.shape
        Ho = (Hi - 1) * stride - 2 * padding + kH
        Wo = (Wi - 1) * stride - 2 * padding + kW
        y = torch.empty((N, Co, Ho, Wo), device=x.device, dtype=torch.float32)
        # "convolution" view: input = y-shaped (N,Co,1,Ho,Wo), output = x-shaped (N,Ci,1,Hi,Wi), weight (Ci,Co,1,kH,kW)
        y5, x5, w5 = y.unsqueeze(2), x.unsqueeze(2), weight.unsqueeze(2)
        d = _conv_desc(y5, w5, x5, (1, stride, stride), (0, padding, padding))
        _call("cvad_conv_dgrad_f32", ctypes.byref(d), _ptr(x5), _ptr(weight), _ptr(y5), 0, _st())
        ctx.geom = (stride, padding)
        ctx.weight = weight
        ctx.save_for_backward(x)
        return y

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        stride, padding = ctx.geom
        weight = ctx.weight
        dy = _f32c(dy)
        dy5, x5, w5 = dy.unsqueeze(2), x.unsqueeze(2), weight.unsqueeze(2)
        dx = None
        if ctx.needs_input_grad[0]:
            dx5 = torch.empty(x5.shape, device=x.device, dtype=torch.float32)
            d = _conv_desc(dy5, w5, dx5, (1, stride, stride), (0, padding, padding))
            _call("cvad_conv_fwd_f32", ctypes.byref(d), _ptr(dy5), _ptr(weight), None, _ptr(dx5), ACT_NONE, _st())
            dx = dx5.squeeze(2)
        if _wants_grad(weight):
            d = _conv_desc(dy5, w5, x5, (1, stride, stride), (0, padding, padding))
            _call("cvad_conv_wgrad_f32", ctypes.byref(d), _ptr(dy5), _ptr(x5), _ptr(grad_buffer(weight)), _st())
        return dx, None, None, None


def conv_transpose2d(x, weight, stride, padding):
    return _ConvTranspose2d.apply(x, weight, stride, padding)


class _ChannelBiasAct(torch.autograd.Function):
    """y = act(x + bias[c]) on (N,C,H,W): the BatchNorm apply / backward kernels with mean 0, invstd 1, gamma 1."""

    @staticmethod
    def forward(ctx, x, bias, act):
        _cuda(x, bias)
        x = _f32c(x)
        N, C = x.shape[:2]
        S = x[0, 0].numel()
        zeros = torch.zeros(C, device=x.device, dtype=torch.float32)
        ones = torch.ones(C, device=x.device, dtype=torch.float32)
        y = torch.empty_like(x)
        _call("cvad_bn_apply_f32", _ptr(x), _ptr(y), N, C, S, _ptr(zeros), _ptr(ones), _ptr(ones), _ptr(bias), act, _st())
        ctx.meta = act
        ctx.bias = bias
        ctx.save_for_backward(x, zeros, ones)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, zeros, ones = ctx.saved_tensors
        bias, act = ctx.bias, ctx.meta
        dy = _f32c(dy)
        N, C = x.shape[:2]
        S = x[0, 0].numel()
        dx = torch.empty_like(x)
        db = grad_buffer(bias) if _wants_grad(bias) else None
        _call("cvad_bn_bwd_f32", _ptr(dy), _ptr(x), _ptr(dx), N, C, S, _ptr(zeros), _ptr(ones), _ptr(ones), _ptr(bias), act, 0,
              _ptr(bn_workspace(x.device, C)), None, _ptr(db), _st())
        return dx, None, None


def channel_bias_act(x, bias, act=ACT_NONE):
    return _ChannelBiasAct.apply(x, bias, act)


class _LstmLast(torch.autograd.Function):
    """Last hidden state of nn.LSTM(64->64) given the precomputed input projection gi (N,T,256) (cad1:238-239)."""

    @staticmethod
    def forward(ctx, gi, w_hh, b_hh):
        _cuda(gi, w_hh, b_hh)
        gi = _f32c(gi)
        N, T, _ = gi.shape
        hT = torch.empty((N, 64), device=gi.device, dtype=torch.float32)
        need = ctx.needs_input_grad[0] or w_hh.requires_grad
        saved = torch.empty((N, T, 6, 64), device=gi.device, dtype=torch.float32) if need else None
        _call("cvad_lstm_fwd_f32", _ptr(gi), _ptr(w_hh), _ptr(b_hh), N, T, _ptr(hT), _ptr(saved), _st())
        ctx.w_hh, ctx.b_hh, ctx.shape = w_hh, b_hh, (N, T)
        ctx.save_for_backward(saved)
        return hT

    @staticmethod
    def backward(ctx, dhT):
        (saved,) = ctx.saved_tensors
        N, T = ctx.shape
        w_hh, b_hh = ctx.w_hh, ctx.b_hh
        dgi = torch.empty((N, T, 256), device=dhT.device, dtype=torch.float32)
        dw = grad_buffer(w_hh) if _wants_grad(w_hh) else None
        db = grad_buffer(b_hh) if _wants_grad(b_hh) else None
        _call("cvad_lstm_bwd_f32", _ptr(_f32c(dhT)), _ptr(saved), _ptr(w_hh), N, T, _ptr(dgi), _ptr(dw), _ptr(db), _st())
        return dgi, None, None


def lstm_last(gi, w_hh, b_hh):
    return _LstmLast.apply(gi, w_hh, b_hh)


class _ReconMse(torch.autograd.Function):
    """mean((recon - frames)^2) (cad1:323-344) where recon is (B,T,E) or one reconstruction per clip (B,E) broadcast over T.
    Returns (loss, per-clip mean error (B,))."""

    @staticmethod
    def forward(ctx, recon, frames, flag):
        _cuda(recon, frames)
        frames = _f32c(frames)
        B, T = frames.shape[:2]
        E = frames[0, 0].numel()
        recon = _f32c(recon)
        rts = 0 if recon.numel() == B * E else E
        ws = torch.zeros(B, device=frames.device, dtype=torch.float64)
        clip = torch.empty(B, device=frames.device, dtype=torch.float32)
        loss = torch.empty(1, device=frames.device, dtype=torch.float32)
        dr = torch.empty_like(recon) if ctx.needs_input_grad[0] else None
        _call("cvad_recon_mse_f32", _ptr(recon), rts, _ptr(frames), B, T, E, _ptr(ws), _ptr(clip), _ptr(loss), _ptr(dr), _ptr(flag), _st())
        ctx.save_for_backward(dr)
        ctx.mark_non_differentiable(clip)
        return loss[0], clip

    @staticmethod
    def backward(ctx, g, _g2):
        (dr,) = ctx.saved_tensors
        return dr * g, None, None


def recon_mse(recon, frames, flag=None):
    return _ReconMse.apply(recon, frames, flag)


def memory_score(seq, memory, n_filled):
    """cad1:262-301 (no gradient: the score is an evaluation signal)."""
    _cuda(seq, memory)
    seq = _f32c(seq.detach())
    B, D = seq.shape
    out = torch.zeros(B, device=seq.device, dtype=torch.float32)
    if n_filled >= 10:
        _call("cvad_memory_score_f32", _ptr(seq), _ptr(memory), B, int(n_filled), D, _ptr(out), _st())
    return out
