"""The BatchNorm + ReLU kernels of the bf16 backbone (csrc/nhwc_bf16.cu) against a plain fp64 reference, entry by entry as tc.py chains
them: at every BatchNorm shape of the benchmarked step (512 frames of 240x360), at edge shapes, with the workspace shared across calls, and
under every development knob of the apply kernels (each in a child process: the knobs are read once per process).

Every check prints its observed error next to its bound; each bound is derived from the kernel's arithmetic where it is stated.

    python tests/test_bn_flat_gpu.py --child out.pt     # the knob subset of one process (the knob settings come from the environment)
"""
import math
import os
import subprocess
import sys
import tempfile

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 2.0 ** -24                  # fp32 unit roundoff: |fl(v) - v| <= U |v|
EPS, MOM = 1e-5, 0.1
BF16 = torch.bfloat16
LAMBDA = 4.0                    # probabilistic rounding-error bound of a k-term fp32 sum: lambda * sqrt(k) * U * sum|terms| (Higham & Mary, 2019)


# ------------------------------------------------------------------------------------------------ fp64 reference (device-agnostic)
def _c(v):
    return v.view(1, -1, 1, 1)


def ref_stats(x):
    """x (N, C, H, W) fp64 -> batch mean, biased variance, invstd, unbiased variance."""
    n = x.numel() // x.shape[1]
    m = x.mean(dim=(0, 2, 3))
    v = (x - _c(m)).square().mean(dim=(0, 2, 3))
    return m, v, 1.0 / torch.sqrt(v + EPS), (v * n / (n - 1) if n > 1 else v)


def ref_running(r0, stat):
    return (1.0 - MOM) * r0 + MOM * stat


def ref_forward(x, gamma, beta, m, invstd):
    """relu(x a + b), a = gamma invstd, b = beta - m a.  Returns act, pre-activation, a, b (fp64)."""
    a = gamma * invstd
    b = beta - m * a
    pre = x * _c(a) + _c(b)
    return pre.clamp_min(0.0), pre, a, b


def ref_backward(x, dact, gamma, beta, m, invstd, training):
    """ReLU + BatchNorm backward: draw, dgamma, dbeta (and g, xhat, pre) from the mean / invstd the forward used."""
    a = gamma * invstd
    b = beta - m * a
    pre = x * _c(a) + _c(b)
    g = dact * (pre > 0)
    xhat = (x - _c(m)) * _c(invstd)
    dbeta = g.sum(dim=(0, 2, 3))
    dgamma = (g * xhat).sum(dim=(0, 2, 3))
    if training:
        n = x.numel() // x.shape[1]
        draw = _c(a) * (g - _c(dbeta / n) - xhat * _c(dgamma / n))
    else:
        draw = _c(a) * g
    return draw, dgamma, dbeta, g, xhat, pre


@pytest.mark.parametrize("training", [True, False])
def test_reference_matches_torch_batch_norm(training):
    """The fp64 reference above against F.batch_norm + relu and autograd in fp64 (CPU)."""
    gen = torch.Generator().manual_seed(3)
    N, C, H, W = 3, 5, 4, 7
    x = (torch.randn(N, C, H, W, generator=gen, dtype=torch.float64) + _c(torch.arange(C, dtype=torch.float64))) * 1.7
    gamma = torch.randn(C, generator=gen, dtype=torch.float64)
    beta = torch.randn(C, generator=gen, dtype=torch.float64) * 0.3
    dact = torch.randn(N, C, H, W, generator=gen, dtype=torch.float64)
    rm0 = torch.randn(C, generator=gen, dtype=torch.float64)
    rv0 = torch.rand(C, generator=gen, dtype=torch.float64) + 0.5
    rm, rv = rm0.clone(), rv0.clone()
    xr, gr, br = x.clone().requires_grad_(True), gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    y = F.relu(F.batch_norm(xr, rm, rv, gr, br, training, MOM, EPS))
    dx, dg, db = torch.autograd.grad(y, (xr, gr, br), dact)
    if training:
        m, _, invstd, vu = ref_stats(x)
        assert torch.allclose(rm, ref_running(rm0, m), rtol=1e-13, atol=1e-13)
        assert torch.allclose(rv, ref_running(rv0, vu), rtol=1e-13, atol=1e-13)
    else:
        m, invstd = rm0, 1.0 / torch.sqrt(rv0 + EPS)
    act = ref_forward(x, gamma, beta, m, invstd)[0]
    draw, dgamma, dbeta = ref_backward(x, dact, gamma, beta, m, invstd, training)[:3]
    assert torch.allclose(act, y.detach(), rtol=1e-12, atol=1e-12)
    assert torch.allclose(draw, dx, rtol=1e-11, atol=1e-12)
    assert torch.allclose(dgamma, dg, rtol=1e-11, atol=1e-12) and torch.allclose(dbeta, db, rtol=1e-11, atol=1e-12)


# ------------------------------------------------------------------------------------------------ inputs
# (N, H, W, C, phase): every BatchNorm of the benchmarked step -- the output of a layer feeding a stride-2 convolution is written as
# phase planes (tc.act_shape) -- then N = 1 (divisor 1 skips fast_div), ragged N (row count not a multiple of R x grid), odd phase
# geometries, and N = 3 (one row group per CTA)
BENCH_SHAPES = [(512, 60, 90, 32, 0), (512, 60, 90, 32, 1), (512, 30, 45, 64, 0), (512, 30, 45, 64, 1), (512, 15, 23, 128, 0),
                (512, 15, 23, 128, 1), (512, 8, 12, 256, 0)]
EDGE_SHAPES = [(1, 9, 7, 64, 1), (1, 8, 12, 256, 0), (37, 30, 45, 64, 1), (37, 15, 23, 128, 0), (37, 9, 7, 32, 1), (3, 9, 7, 64, 1),
               (3, 12, 18, 32, 1), (3, 15, 23, 128, 0)]
SHAPES = BENCH_SHAPES + EDGE_SHAPES
# the child processes' subset: the largest phase layer, the 256-channel layer, one ragged shape
KNOB_SHAPES = [(512, 60, 90, 32, 1), (512, 8, 12, 256, 0), (37, 15, 23, 128, 0)]
KNOBS = [{}, {"CVAD_BN_ROWS": "4"}, {"CVAD_BN_REVERSE": "0"}, {"CVAD_BN_FOLD": "1"}, {"CVAD_BN_OCC": "3"}, {"CVAD_BN_SMALL_GRID": "0"},
         {"CVAD_BN_SMALL_GRID": "0", "CVAD_BN_CTAS": "1"}]


def _id(shape):
    N, H, W, C, phase = shape
    return f"{N}x{H}x{W}x{C}" + ("-phase" if phase else "")


def _seed(shape, k=0):
    N, H, W, C, phase = shape
    return ((N * 131 + H) * 131 + W) * 131 + C * 7 + phase + 1000003 * k


def make_inputs(dev, shape, seed):
    """Conv-output-like interior x (bf16 values): per-channel offsets up to +-4 sigma, two channels at +-8 sigma, per-channel sigma;
    gammas of both signs; beta ~ 0.5 |gamma| N(0, 1) so that about half of the ReLUs are open; a bf16 upstream gradient dy."""
    N, H, W, C, _ = shape
    gen = torch.Generator(device=dev).manual_seed(seed)
    sigma = 0.25 + 2.0 * torch.rand(C, generator=gen, device=dev)
    off = torch.rand(C, generator=gen, device=dev) * 8.0 - 4.0
    off[3] = 8.0
    off[C - 2] = -8.0
    x = ((torch.randn(N, C, H, W, generator=gen, device=dev) + _c(off)) * _c(sigma)).to(BF16).double()
    gamma = 0.5 + torch.rand(C, generator=gen, device=dev)
    gamma[1::4] *= -1.0
    beta = 0.5 * gamma.abs() * torch.randn(C, generator=gen, device=dev)
    dy = (torch.randn(N, C, H, W, generator=gen, device=dev) * _c(0.5 + torch.rand(C, generator=gen, device=dev))).to(BF16).double()
    # running statistics near the batch's own (as after training), so that eval mode also leaves about half of the ReLUs open
    rm0 = (off + 0.2 * torch.randn(C, generator=gen, device=dev)) * sigma
    rv0 = sigma.square() * (0.8 + 0.4 * torch.rand(C, generator=gen, device=dev))
    # dgamma / dbeta arrive holding a non-zero value (the kernels accumulate with +=)
    dg0 = 100.0 * (1.0 + torch.rand(C, generator=gen, device=dev))
    db0 = -100.0 * (1.0 + torch.rand(C, generator=gen, device=dev))
    return dict(x=x, gamma=gamma, beta=beta, dy=dy, rm0=rm0, rv0=rv0, dg0=dg0, db0=db0)


def _raw(x):
    from cvad_b200 import tc
    raw = tc.to_padded(x.float())
    raw[:, 0] = 9.0                      # convolution outputs carry junk in their border
    raw[:, :, 0] = -9.0
    raw[:, -1] = 5.0
    raw[:, :, -1] = 3.0
    return raw


def _dact(dy, phase):
    from cvad_b200 import tc
    if phase:
        return tc.to_phase(dy.float())
    d = tc.to_padded(dy.float())
    d[:, 0] = 11.0                       # data-gradients carry junk in their border as well
    d[:, :, -1] = -4.0
    return d


def _nan(shape, dev, dtype=BF16):
    return torch.full(shape if isinstance(shape, tuple) else (shape,), float("nan"), device=dev, dtype=dtype)


def _exact_sums(x):
    return torch.cat([x.sum(dim=(0, 2, 3)), x.square().sum(dim=(0, 2, 3))])


# ------------------------------------------------------------------------------------------------ entry chains (as tc.py calls them)
def _ws(dev, C):
    from cvad_b200 import ops
    return ops.bn_workspace(dev, C)


def run_forward_fused(dev, shape, inp):
    """Training forward, default path: ws holds the exact fp64 sums (the convolution epilogue's contract), then finalize + apply."""
    from cvad_b200 import tc
    from cvad_b200.ops import _call, _ptr, _st
    N, H, W, C, phase = shape
    raw = _raw(inp["x"])
    ws = _ws(dev, C)
    ws.copy_(_exact_sums(inp["x"]))
    act = _nan(tc.act_shape(N, H, W, C, phase), dev)
    mean, invstd = _nan(C, dev, torch.float32), _nan(C, dev, torch.float32)
    rm, rv, nbt = inp["rm0"].clone(), inp["rv0"].clone(), torch.tensor(5, device=dev)
    _call("cvad_pad_bn_finalize_apply_relu_bf16", _ptr(raw), _ptr(act), N, H, W, C, phase, _ptr(ws), EPS, MOM, _ptr(inp["gamma"]),
          _ptr(inp["beta"]), _ptr(mean), _ptr(invstd), _ptr(rm), _ptr(rv), _ptr(nbt), _st())
    return dict(act=act, mean=mean, invstd=invstd, rm=rm, rv=rv, nbt=nbt, ws=ws.clone())


def run_forward_unfused(dev, shape, inp):
    """Training forward, unfused: the reduce kernel's statistics, then the apply."""
    from cvad_b200 import tc
    from cvad_b200.ops import _call, _ptr, _st
    N, H, W, C, phase = shape
    raw = _raw(inp["x"])
    ws = _ws(dev, C)
    mean, invstd = _nan(C, dev, torch.float32), _nan(C, dev, torch.float32)
    rm, rv, nbt = inp["rm0"].clone(), inp["rv0"].clone(), torch.tensor(5, device=dev)
    _call("cvad_pad_bn_stats_bf16", _ptr(raw), N, H, W, C, _ptr(ws), EPS, MOM, _ptr(mean), _ptr(invstd), _ptr(rm), _ptr(rv), _ptr(nbt), _st())
    out = dict(mean=mean, invstd=invstd, rm=rm, rv=rv, nbt=nbt, ws=ws.clone())
    act = _nan(tc.act_shape(N, H, W, C, phase), dev)
    _call("cvad_pad_bn_apply_relu_bf16", _ptr(raw), _ptr(act), N, H, W, C, phase, _ptr(mean), _ptr(invstd), _ptr(inp["gamma"]),
          _ptr(inp["beta"]), _st())
    out["act"] = act
    return out


def run_forward_eval(dev, shape, inp):
    from cvad_b200 import tc
    from cvad_b200.ops import _call, _ptr, _st
    N, H, W, C, phase = shape
    raw = _raw(inp["x"])
    mean, invstd = _nan(C, dev, torch.float32), _nan(C, dev, torch.float32)
    _call("cvad_bn_eval_prepare_f32", C, EPS, _ptr(inp["rm0"]), _ptr(inp["rv0"]), _ptr(mean), _ptr(invstd), _st())
    act = _nan(tc.act_shape(N, H, W, C, phase), dev)
    _call("cvad_pad_bn_apply_relu_bf16", _ptr(raw), _ptr(act), N, H, W, C, phase, _ptr(mean), _ptr(invstd), _ptr(inp["gamma"]),
          _ptr(inp["beta"]), _st())
    return dict(act=act, mean=mean, invstd=invstd)


def backward_stats(dev, inp, training):
    """The fp32 mean / invstd the backward receives: the forward's batch statistics (fp64 reference rounded to fp32), or in eval mode
    what cvad_bn_eval_prepare_f32 makes of the running statistics."""
    from cvad_b200.ops import _call, _ptr, _st
    if training:
        m, _, invstd, _ = ref_stats(inp["x"])
        return m.float(), invstd.float()
    C = inp["x"].shape[1]
    mean, invstd = _nan(C, dev, torch.float32), _nan(C, dev, torch.float32)
    _call("cvad_bn_eval_prepare_f32", C, EPS, _ptr(inp["rm0"]), _ptr(inp["rv0"]), _ptr(mean), _ptr(invstd), _st())
    return mean, invstd


def run_backward(dev, shape, inp, training, fused=True):
    """Backward, default path (reduce + apply + parameter update) with dgamma / dbeta pre-filled, again with both null (frozen
    parameters), and -- training only -- the fused path: ws seeded with the exact sum g / sum g*xhat, then apply + parameter update."""
    from cvad_b200.ops import _call, _ptr, _st
    N, H, W, C, phase = shape
    raw, dact = _raw(inp["x"]), _dact(inp["dy"], phase)
    mean, invstd = backward_stats(dev, inp, training)
    ws = _ws(dev, C)
    out = dict(mean=mean, invstd=invstd)
    args = (N, H, W, C, phase, _ptr(mean), _ptr(invstd), _ptr(inp["gamma"]), _ptr(inp["beta"]), int(training), _ptr(ws))
    draw, dg, db = _nan(raw.shape, dev), inp["dg0"].clone(), inp["db0"].clone()
    _call("cvad_pad_bn_relu_bwd_bf16", _ptr(raw), _ptr(dact), _ptr(draw), *args, _ptr(dg), _ptr(db), _st())
    out.update(draw=draw, dg=dg, db=db, ws=ws.clone())
    draw = _nan(raw.shape, dev)
    _call("cvad_pad_bn_relu_bwd_bf16", _ptr(raw), _ptr(dact), _ptr(draw), *args, None, None, _st())
    out.update(draw_np=draw, ws_np=ws.clone())
    if training and fused:
        _, dgamma, dbeta = ref_backward(inp["x"], inp["dy"], inp["gamma"], inp["beta"], mean.double(), invstd.double(), True)[:3]
        ws.copy_(torch.cat([dbeta, dgamma]))
        draw, dg, db = _nan(raw.shape, dev), inp["dg0"].clone(), inp["db0"].clone()
        _call("cvad_pad_bn_relu_bwd_apply_bf16", _ptr(raw), _ptr(dact), _ptr(draw), *args, _ptr(dg), _ptr(db), _st())
        out.update(draw_f=draw, dg_f=dg, db_f=db, ws_f=ws.clone())
    return out


# ------------------------------------------------------------------------------------------------ checks
def _ratio(err, bound):
    return torch.where(err == 0, 0.0, err / bound)          # a zero bound admits only a zero error


def _report(label, err_over_bound, detail=""):
    r = float(err_over_bound)
    print(f"[bn] {label}: err/bound {r:.3f}{detail}")
    assert r <= 1.0, f"{label}: error exceeds its bound by {r:.3f}x{detail}"


def _check_ws(label, ws):
    assert float(ws.abs().max()) == 0.0, f"{label}: the workspace is not zero after the call"


def reduce_run_length(shape, bwd):
    """Longest run of pixels one thread of pad_reduce_kernel sums in fp32 (launch_reduce: one wave of 4 forward / 3 backward CTAs per SM,
    each CTA a contiguous chunk of the N*H*W pixels over its 2048/C pixel slots)."""
    N, H, W, C, _ = shape
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    blocks = min(N * H, (3 if bwd else 4) * sms)
    chunk = -(-(N * H * W) // blocks)
    return -(-chunk // (2048 // C))


def check_act(label, shape, act, x, gamma, beta, m, invstd):
    """act vs relu(x a + b) from (m, invstd) in fp64.
    Bound: the kernel's pre-activation fma(x, sc, sh), sc = fl(invstd32 gamma), sh = fl(beta - mu32 sc), is off by at most
    |x a| (eps + 2 U) + |m a| (eps + 4 U) + 2 U |b| with eps <= 2.5 U the relative error of the fp32 mean / invstd it was given (one
    rounding from the exact sums, three in cvad_bn_eval_prepare_f32): <= 6.5 U (|x a| + |m a| + |b|), held by 1e-6 (17 U) x the same.
    |m a| belongs in it: where beta ~ m a, b is tiny while the rounding of sh is not (pre-activations of ~1e-6 from |x a| ~ 1e-3 showed it).
    The bf16 store (8-bit significand) then adds up to 2^-8 |v|.  Borders and phase holes are exact zeros, and no NaN of the pre-fill
    survives."""
    from cvad_b200 import tc
    N, H, W, C, phase = shape
    assert not bool(torch.isnan(act).any()), f"{label}: act has elements the kernel did not write"
    got = tc.from_phase(act, H, W) if phase else tc.from_padded(act, H, W)
    ref, pre, a, b = ref_forward(x, gamma.double(), beta.double(), m.double(), invstd.double())
    bound = 2.0 ** -8 * ref + 1e-6 * ((x * _c(a)).abs() + _c((m.double() * a).abs() + b.abs()))
    del pre
    err = (got.double() - ref).abs()
    _report(f"{label} act", _ratio(err, bound).max(), f" (max |err| {float(err.max()):.2e})")
    del err, bound, ref
    ones = torch.ones(1, 1, H, W, device=act.device)
    filled = (tc.to_phase(ones) if phase else tc.to_padded(ones)) != 0
    holes = act.masked_fill(filled, 0.0)
    assert float(holes.float().abs().max()) == 0.0, f"{label}: border / phase holes of act are not zero"


def check_stats(label, shape, out, x, rm0, rv0, exact):
    """mean / invstd / running statistics / num_batches_tracked vs fp64.
    exact (finalize from the exact fp64 sums): m and var in fp64 (relative error ~1e-14 even at 8 sigma: 65 x 2^-53), then one fp32 rounding
    each -> |err| <= U |ref|; bound 2 U |ref|.
    reduce kernel: each thread sums a run of k pixels in fp32 (sum x, fma sum x^2), combined in fp64: |d sum x| <= LAMBDA sqrt(k) U sum|x|,
    |d sum x^2| <= LAMBDA sqrt(k) U sum x^2 -> |d m| <= LAMBDA sqrt(k) U E|x|, |d var| <= LAMBDA sqrt(k) U (E x^2 + 2 |m| E|x|),
    |d invstd| / invstd <= |d var| / (2 (var + eps)); plus the fp32 rounding of the result.
    Running statistics: (1 - mom) r0 + mom stat in fp32 (momentum 0.1f): <= 4 U (0.9 |r0| + 0.1 |stat|) + 0.1 |d stat|."""
    N, H, W, C, _ = shape
    m, v, invstd, vu = ref_stats(x)
    if exact:
        dm, dis = 2 * U * m.abs(), 2 * U * invstd
    else:
        k = reduce_run_length(shape, False)
        ex, ex2 = x.abs().mean(dim=(0, 2, 3)), x.square().mean(dim=(0, 2, 3))
        s = LAMBDA * math.sqrt(k) * U
        dv = s * (ex2 + 2 * m.abs() * ex)
        dm = U * m.abs() + s * ex
        dis = U * invstd + invstd * dv / (2 * (v + EPS))
    tag = "exact sums" if exact else f"reduce, k = {reduce_run_length(shape, False)}"
    _report(f"{label} mean ({tag})", ((out["mean"].double() - m).abs() / dm).max(),
            f" (max |err| / (U |m|) {float(((out['mean'].double() - m).abs() / (U * m.abs())).max()):.2f})")
    _report(f"{label} invstd ({tag})", ((out["invstd"].double() - invstd).abs() / dis).max(),
            f" (max |err| / (U invstd) {float(((out['invstd'].double() - invstd).abs() / (U * invstd)).max()):.2f})")
    dvu = dis / invstd * 2 * (vu + EPS)          # |d var| back from the invstd bound
    for name, key, r0, stat, dstat in (("running_mean", "rm", rm0, m, dm), ("running_var", "rv", rv0, vu, dvu)):
        bound = 4 * U * (0.9 * r0.double().abs() + 0.1 * stat.abs()) + 0.1 * dstat
        _report(f"{label} {name}", ((out[key].double() - ref_running(r0.double(), stat)).abs() / bound).max())
    assert int(out["nbt"]) == 6, f"{label}: num_batches_tracked {int(out['nbt'])}, expected 6"
    _check_ws(label, out["ws"])


def check_backward(label, shape, out, inp, training, exact_sums, dg, db, draw):
    """draw / dgamma / dbeta vs the fp64 backward at the fp32 mean / invstd the kernel received.
    draw: the kernel forms a g - k0 - k1 x with fp32 constants ca = fl(gamma invstd), k1 = fl(fl(ca mgx) invstd), k0 = fl(ca mg - k1 mu)
    (mg, mgx = fp32 means of the two sums): each term carries a few U of its own magnitude, |a g|, |a mg| <= max|a g| and
    |k1 x| <= |a| |mgx| |x invstd| <= 12 max|a g| here, so the pre-rounding error stays below ~60 U max_c|a g| < 1e-5 max_c|a g|;
    the bf16 store adds up to 2^-8 |v|.  Elements whose pre-activation lies within the fp32 rounding of the gate
    (8 U (|x a| + |b| + |beta|)) may take the other ReLU branch in the kernel: they are left out and counted.  The border is exactly 0.
    dbeta / dgamma: fp32 rounding of the fp64 sum and of the += (U |S| + U |D0 + S|, bound x 1.01) -- plus, when the reduce kernel took the
    sums, its fp32 per-thread runs of k pixels: LAMBDA sqrt(k) U sum|g| for sum g, and for sum g xhat = invstd (sum g x - m sum g):
    LAMBDA sqrt(k) U invstd (sum|g x| + |m| sum|g|)."""
    N, H, W, C, phase = shape
    x, gamma, beta = inp["x"], inp["gamma"].double(), inp["beta"].double()
    m, invstd = out["mean"].double(), out["invstd"].double()
    ref, dgamma, dbeta, g, xhat, pre = ref_backward(x, inp["dy"], gamma, beta, m, invstd, training)
    a, b = gamma * invstd, beta - m * gamma * invstd
    near = pre.abs() <= 8 * U * ((x * _c(a)).abs() + _c(b.abs() + beta.abs()))
    del pre
    assert not bool(torch.isnan(draw).any()), f"{label}: draw has elements the kernel did not write"
    got = draw[:, 1:H + 1, 1:W + 1, :].permute(0, 3, 1, 2).double()
    scale = (g * _c(a)).abs().amax(dim=(0, 2, 3))
    bound = 2.0 ** -8 * ref.abs() + 1e-5 * _c(scale)
    ratio = _ratio((got - ref).abs(), bound).masked_fill(near, 0.0)
    _report(f"{label} draw", ratio.max(), f" ({int(near.sum())} elements at the ReLU edge left out)")
    del ratio, bound, got, ref
    border = draw.clone()
    border[:, 1:H + 1, 1:W + 1] = 0
    assert float(border.float().abs().max()) == 0.0, f"{label}: border of draw is not zero"
    if dg is None:
        return
    t_b, t_g = 0.0, 0.0
    if not exact_sums:
        s = LAMBDA * math.sqrt(reduce_run_length(shape, True)) * U
        t_b = s * g.abs().sum(dim=(0, 2, 3))
        t_g = s * invstd * ((g * x).abs().sum(dim=(0, 2, 3)) + m.abs() * g.abs().sum(dim=(0, 2, 3)))
    for name, got_p, d0, S, t in (("dbeta", db, inp["db0"], dbeta, t_b), ("dgamma", dg, inp["dg0"], dgamma, t_g)):
        want = d0.double() + S
        bound = 1.01 * U * (S.abs() + want.abs()) + t
        err = (got_p.double() - want).abs()
        _report(f"{label} {name}", _ratio(err, bound).max(), f" (max |err| / sum|g| {float((err / g.abs().sum(dim=(0, 2, 3))).max()):.1e})")


def check_forward_fused(label, shape, inp, out):
    m, _, invstd, _ = ref_stats(inp["x"])
    check_stats(label, shape, out, inp["x"], inp["rm0"], inp["rv0"], exact=True)
    check_act(label, shape, out["act"], inp["x"], inp["gamma"], inp["beta"], m, invstd)


def check_forward_unfused(label, shape, inp, out):
    check_stats(label, shape, out, inp["x"], inp["rm0"], inp["rv0"], exact=False)
    # act against the statistics the apply was given (their own error is bounded above)
    check_act(label, shape, out["act"], inp["x"], inp["gamma"], inp["beta"], out["mean"], out["invstd"])


def check_backward_all(label, shape, inp, out, training):
    check_backward(f"{label} default", shape, out, inp, training, False, out["dg"], out["db"], out["draw"])
    _check_ws(f"{label} default", out["ws"])
    check_backward(f"{label} frozen parameters", shape, out, inp, training, False, None, None, out["draw_np"])
    _check_ws(f"{label} frozen parameters", out["ws_np"])
    if "draw_f" in out:
        check_backward(f"{label} fused sums", shape, out, inp, training, True, out["dg_f"], out["db_f"], out["draw_f"])
        _check_ws(f"{label} fused sums", out["ws_f"])


# ------------------------------------------------------------------------------------------------ workspace reuse
# stream-ordered calls that share ops.bn_workspace (one per width) and the reduce kernel's module-global replicas / ticket:
# layer1's two BatchNorms (same C, different inputs); a C = 256 reduce followed by a C = 32 one; forward statistics of one layer
# between backward reduces of others (one of them the same width); a fused backward and a finalize in between
WS_SEQUENCE = [("stats", (64, 30, 45, 32, 0), 1), ("stats", (64, 30, 45, 32, 0), 2), ("stats", (64, 8, 12, 256, 0), 3),
               ("stats", (64, 30, 45, 32, 0), 4), ("backward", (37, 30, 45, 64, 0), 5), ("stats", (37, 30, 45, 64, 1), 6),
               ("backward", (37, 15, 23, 128, 1), 7), ("finalize", (37, 30, 45, 64, 0), 8), ("backward", (37, 30, 45, 64, 1), 9),
               ("stats", (64, 8, 12, 256, 0), 10)]


def run_ws_sequence(dev):
    outs = []
    for kind, shape, k in WS_SEQUENCE:
        inp = make_inputs(dev, shape, _seed(shape, k))
        if kind == "stats":
            outs.append(run_forward_unfused(dev, shape, inp))
        elif kind == "finalize":
            outs.append(run_forward_fused(dev, shape, inp))
        else:
            outs.append(run_backward(dev, shape, inp, True, fused=(k == 9)))
    return outs


def check_ws_sequence(dev, outs, tag=""):
    for i, ((kind, shape, k), out) in enumerate(zip(WS_SEQUENCE, outs)):
        inp = make_inputs(dev, shape, _seed(shape, k))
        label = f"{tag}ws#{i} {kind} {shape}"
        if kind == "stats":
            check_forward_unfused(label, shape, inp, out)
        elif kind == "finalize":
            check_forward_fused(label, shape, inp, out)
        else:
            check_backward_all(label, shape, inp, out, True)


# ------------------------------------------------------------------------------------------------ GPU tests
def _fresh(dev, C):
    _ws(dev, C).zero_()          # a failed earlier case must not leak into this one


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=_id)
def test_bn_forward_training(dev, shape):
    inp = make_inputs(dev, shape, _seed(shape))
    _fresh(dev, shape[3])
    check_forward_fused(f"fwd {shape}", shape, inp, run_forward_fused(dev, shape, inp))
    check_forward_unfused(f"fwd unfused {shape}", shape, inp, run_forward_unfused(dev, shape, inp))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=_id)
def test_bn_forward_eval(dev, shape):
    inp = make_inputs(dev, shape, _seed(shape))
    out = run_forward_eval(dev, shape, inp)
    rm, rv = inp["rm0"].double(), inp["rv0"].double()
    assert torch.equal(out["mean"], inp["rm0"])
    # 1.f / sqrtf(rv + eps) in fp32: U from the sum (U / 2 after the square root), U from sqrtf, U from the division
    _report(f"eval {shape} invstd", ((out["invstd"].double() - 1.0 / torch.sqrt(rv + EPS)).abs() / (3 * U / torch.sqrt(rv + EPS))).max())
    check_act(f"eval {shape}", shape, out["act"], inp["x"], inp["gamma"], inp["beta"], rm, 1.0 / torch.sqrt(rv + EPS))


@pytest.mark.gpu
@pytest.mark.parametrize("shape,training", [(s, True) for s in SHAPES] + [(BENCH_SHAPES[1], False), (EDGE_SHAPES[3], False)],
                         ids=[_id(s) + "-training" for s in SHAPES] + [_id(BENCH_SHAPES[1]) + "-eval", _id(EDGE_SHAPES[3]) + "-eval"])
def test_bn_backward(dev, shape, training):
    inp = make_inputs(dev, shape, _seed(shape))
    _fresh(dev, shape[3])
    out = run_backward(dev, shape, inp, training)
    check_backward_all(f"bwd {shape} {'training' if training else 'eval'}", shape, inp, out, training)


@pytest.mark.gpu
def test_bn_workspace_reuse(dev):
    for C in (32, 64, 128, 256):
        _fresh(dev, C)
    check_ws_sequence(dev, run_ws_sequence(dev))


# ------------------------------------------------------------------------------------------------ knob variants (child processes)
def run_child(dev):
    """The knob subset: training forward (both paths) and backward (all three) at KNOB_SHAPES, then the workspace sequence."""
    res = {}
    for shape in KNOB_SHAPES:
        _fresh(dev, shape[3])
        inp = make_inputs(dev, shape, _seed(shape))
        res[shape] = dict(fwd=run_forward_fused(dev, shape, inp), fwd_unfused=run_forward_unfused(dev, shape, inp),
                          bwd=run_backward(dev, shape, inp, True))
        torch.cuda.synchronize()
        res[shape] = {k: {n: t.cpu() for n, t in v.items()} for k, v in res[shape].items()}
    for C in (32, 64, 128, 256):
        _fresh(dev, C)
    res["ws"] = [{n: t.cpu() for n, t in o.items()} for o in run_ws_sequence(dev)]
    return res


_DEFAULT = []           # the default setting's results, the yardstick of the bit-identity check


def _child_results(knobs):
    if not knobs and _DEFAULT:
        return _DEFAULT[0]
    env = dict(os.environ)
    for k in ("CVAD_BN_ROWS", "CVAD_BN_REVERSE", "CVAD_BN_FOLD", "CVAD_BN_OCC", "CVAD_BN_SMALL_GRID", "CVAD_BN_CTAS"):
        env.pop(k, None)
    env.update(knobs)
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "out.pt")
        cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), "--child", path]
        r = subprocess.run(cmd, env=env, cwd=ROOT, timeout=900, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert r.returncode == 0, f"child with {knobs} failed:\n{r.stdout[-4000:]}"
        res = torch.load(path)
    if not knobs:
        _DEFAULT.append(res)
    return res


def _to(dev, d):
    return {n: t.to(dev) for n, t in d.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("knobs", KNOBS, ids=[" ".join(f"{k}={v}" for k, v in s.items()) or "default" for s in KNOBS])
def test_bn_knob_variants(dev, knobs):
    base = _child_results({})
    res = _child_results(knobs)
    tag = (" ".join(f"{k}={v}" for k, v in knobs.items()) or "default") + " "
    for shape in KNOB_SHAPES:
        inp = make_inputs(dev, shape, _seed(shape))
        r = res[shape]
        check_forward_fused(f"{tag}fwd {shape}", shape, inp, _to(dev, r["fwd"]))
        check_forward_unfused(f"{tag}fwd unfused {shape}", shape, inp, _to(dev, r["fwd_unfused"]))
        check_backward_all(f"{tag}bwd {shape}", shape, inp, _to(dev, r["bwd"]), True)
        # the apply is elementwise arithmetic from the same constants (and the folded finalize is the separate one's arithmetic):
        # act from the exact sums must not change by a bit under any knob
        for n in ("act", "mean", "invstd", "rm", "rv"):
            assert torch.equal(r["fwd"][n], base[shape]["fwd"][n]), f"{tag}{shape}: {n} differs from the default build's"
    check_ws_sequence(dev, [_to(dev, o) for o in res["ws"]], tag)


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "--child":
        sys.path.insert(0, ROOT)
        dev = torch.device("cuda:0")
        out = run_child(dev)
        torch.save(out, sys.argv[2])
    else:
        sys.exit(__doc__)
