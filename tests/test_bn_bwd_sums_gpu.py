"""The bf16 backbone's one-pass BatchNorm backward (include/cvad_b200.h, cvad_pad_bn_relu_bwd_tsum_bf16) and the three kernels that feed it:
the forward apply's ReLU bitmask, the data-gradient's masked column sum S1 = sum g, and T = sum W*dW from the staged weight gradient.

The two identities it rests on are checked in fp64 on the CPU.  On the GPU the chain runs at the seven shapes of the benchmarked step where a
BatchNorm sits under a 3x3 convolution (512 frames; the stride-2 ones put the activation in phase planes).  Every bound is derived from the
arithmetic and printed next to the observed error as a fraction of it."""
import pytest
import torch
import torch.nn.functional as F

U = 2.0 ** -8            # bf16 unit roundoff (8 significant bits, round to nearest)
E = 2.0 ** -24           # fp32 unit roundoff
# per-thread fp32 accumulation runs of the apply kernel: (rows per resident CTA) x (vectors per thread and row) stays below this at every
# shape here (60x90x32: 31744 rows over >= 296 CTAs x 2 vectors; 8x12x256: 5120 rows x 2)
RUN = 1024


def _g(seed):
    return torch.Generator(device="cpu").manual_seed(seed)


# ------------------------------------------------------------------------------------------------ the identities (fp64, CPU)
@pytest.mark.parametrize("stride,H,W", [(1, 15, 23), (2, 15, 23), (2, 8, 12), (1, 8, 12)])
def test_sum_w_dw_equals_sum_act_dact(stride, H, W):
    """For every input channel c of y = conv(a, W) (zero padding, stride 1 or 2): sum_{o,tap} W*dW = sum_p a*da."""
    a = torch.relu(torch.randn(4, 16, H, W, dtype=torch.float64, generator=_g(1)))
    w = torch.randn(24, 16, 3, 3, dtype=torch.float64, generator=_g(2))
    y = F.conv2d(a, w, stride=stride, padding=1)
    dy = torch.randn(y.shape, dtype=torch.float64, generator=_g(3))
    dw = torch.nn.grad.conv2d_weight(a, w.shape, dy, stride=stride, padding=1)
    da = torch.nn.grad.conv2d_input(a.shape, w, dy, stride=stride, padding=1)
    t1, t2 = (w * dw).sum((0, 2, 3)), (a * da).sum((0, 2, 3))
    assert float((t1 - t2).abs().max() / t2.abs().max()) < 1e-14


def test_bn_relu_backward_from_s1_and_t():
    """draw = invstd * (gamma*g - gamma*S1/n - xhat*(T - beta*S1)/n) with S1 = sum g, T = sum act*dact is torch's ReLU + BatchNorm
    backward, and dgamma = sum g*xhat, dbeta = S1."""
    N, C, H, W = 6, 8, 5, 7
    raw = torch.randn(N, C, H, W, dtype=torch.float64, generator=_g(1), requires_grad=True)
    gamma = torch.randn(C, dtype=torch.float64, generator=_g(2), requires_grad=True)
    beta = torch.randn(C, dtype=torch.float64, generator=_g(3), requires_grad=True)
    act = torch.relu(F.batch_norm(raw, None, None, gamma, beta, training=True, eps=1e-5))
    dact = torch.randn(act.shape, dtype=torch.float64, generator=_g(4))
    act.backward(dact)
    n = N * H * W
    x = raw.detach()
    mean = x.mean((0, 2, 3), keepdim=True)
    invstd = (x.var((0, 2, 3), unbiased=False, keepdim=True) + 1e-5).rsqrt()
    xhat = (x - mean) * invstd
    g = dact * (act.detach() > 0)
    s1, t = g.sum((0, 2, 3), keepdim=True), (act.detach() * dact).sum((0, 2, 3), keepdim=True)
    ga, be = gamma.detach().view(1, C, 1, 1), beta.detach().view(1, C, 1, 1)
    draw = invstd * (ga * g - ga * s1 / n - xhat * (t - be * s1) / n)
    assert float((draw - raw.grad).abs().max() / raw.grad.abs().max()) < 1e-13
    assert float(((g * xhat).sum((0, 2, 3)) - gamma.grad).abs().max()) < 1e-12
    assert float((s1.flatten() - beta.grad).abs().max()) < 1e-12


# ------------------------------------------------------------------------------------------------ the chain on the GPU
# (N, H, W, Cin, Cout, stride) of the convolution ABOVE the BatchNorm under test: H x W x Cin is that BatchNorm's activation
CHAIN = [(512, 60, 90, 32, 32, 1), (512, 60, 90, 32, 64, 2), (512, 30, 45, 64, 64, 1), (512, 30, 45, 64, 128, 2),
         (512, 15, 23, 128, 128, 1), (512, 15, 23, 128, 256, 2), (512, 8, 12, 256, 256, 1)]


def _report(label, frac):
    frac = float(frac)
    print(f"[bn-bwd-sums] {label}: max error / bound = {frac:.3f}")
    assert frac <= 1.0, f"{label}: error exceeds its bound ({frac:.3f})"


def _bits(mask, shape):
    """The mask bytes unpacked to one 0/1 value per element of act (byte k = the 8 channels of act's 16-byte vector k)."""
    sh = torch.arange(8, device=mask.device, dtype=torch.uint8)
    return ((mask.view(-1, 1) >> sh) & 1).view(shape)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CHAIN, ids=lambda c: "x".join(map(str, c)))
def test_bn_backward_from_conv_sums(dev, case):
    from cvad_b200 import ops, tc
    from cvad_b200.ops import _call, _ptr, _st
    N, H, W, C, Co, s = case
    phase = s == 2
    Ho, Wo = tc.out_hw(H, W, s)
    n = N * H * W
    # ---- the layer below: raw (junk border), BatchNorm constants with about half the ReLUs open and some negative gammas
    rawf = (torch.randn(N, C, H, W, generator=_g(11)) * 1.5 + 0.3).to(dev).to(torch.bfloat16).float()
    raw = tc.to_padded(rawf)
    raw[:, 0] = 9.0
    raw[:, :, -1] = -5.0
    gamma = (torch.rand(C, generator=_g(12)) + 0.5).to(dev)
    gamma[::5] *= -1.0
    beta = (torch.randn(C, generator=_g(13)) * 0.3).to(dev)
    mean = (torch.randn(C, generator=_g(14)) * 0.2 + 0.3).to(dev)
    invstd = (torch.rand(C, generator=_g(15)) * 0.5 + 0.4).to(dev)
    shape = tc.act_shape(N, H, W, C, phase)
    act = torch.full(shape, 3.0, device=dev, dtype=torch.bfloat16)
    mask = torch.full((act.numel() // 8,), 0xFF, device=dev, dtype=torch.uint8)
    _call("cvad_pad_bn_apply_relu_mask_bf16", _ptr(raw), _ptr(act), _ptr(mask), N, H, W, C, int(phase), _ptr(mean), _ptr(invstd), _ptr(gamma),
          _ptr(beta), _st())
    act0 = torch.empty_like(act)
    _call("cvad_pad_bn_apply_relu_bf16", _ptr(raw), _ptr(act0), N, H, W, C, int(phase), _ptr(mean), _ptr(invstd), _ptr(gamma), _ptr(beta), _st())
    torch.cuda.synchronize()
    assert torch.equal(act, act0), "the mask output changed act"
    bits = _bits(mask, shape)
    assert torch.equal(bits.bool(), act > 0), "mask bit != (act > 0)"
    ones = torch.ones(N, C, H, W, device=dev)
    interior = (tc.to_phase(ones) if phase else tc.to_padded(ones)) > 0
    assert int(bits[~interior].sum()) == 0, "mask bit set on a border / empty plane position"
    del act0, ones

    # ---- the convolution above: draw (zero border) and its weights
    w = (torch.randn(Co, C, 3, 3, generator=_g(16)) / (3.0 * C ** 0.5)).to(dev)
    wd = torch.empty(9 * C, Co, device=dev, dtype=torch.bfloat16)
    _call("cvad_flat_pack_w3x3_bf16", _ptr(w), Co, C, s, None, _ptr(wd), _st())
    dy = tc.to_padded(torch.randn(N, Co, Ho, Wo, generator=_g(17)).to(dev))
    ws = ops.bn_workspace(dev, C)
    ws.zero_()
    # S1: the masked-sum data-gradient writes the same dx as the plain one
    dx0 = torch.full(shape, 7.0, device=dev, dtype=torch.bfloat16)
    dact = torch.full(shape, 7.0, device=dev, dtype=torch.bfloat16)
    _call("cvad_flat_conv3x3_dgrad_bf16", _ptr(dy), _ptr(wd), _ptr(dx0), N, H, W, C, Co, s, _st())
    _call("cvad_flat_conv3x3_dgrad_masksum_bf16", _ptr(dy), _ptr(wd), _ptr(dact), N, H, W, C, Co, s, _ptr(mask), _ptr(ws), _st())
    torch.cuda.synchronize()
    assert torch.equal(dx0, dact), "masked-sum dgrad: dx differs from the plain data-gradient"
    del dx0
    g = (dact.double() * bits).reshape(-1, C)
    s1_ref, sabs = g.sum(0), g.abs().sum(0)
    # fp32 column sums of <= 128 x 8 rows per warp and tile run, then fp64: 1024 E relative to sum |g| covers it
    _report(f"{case} S1", ((ws[:C] - s1_ref).abs() / (RUN * E * sabs + 1e-30)).max())
    # T: the staged weight gradient adds sum bf16(W)*dW of this call; dW itself as from the plain staged entry
    dw, dw0 = torch.zeros(Co, C, 3, 3, device=dev), torch.zeros(Co, C, 3, 3, device=dev)
    scratch = torch.zeros(9 * Co * C, device=dev)
    _call("cvad_flat_conv3x3_wgrad_staged_wdot_bf16", _ptr(act), _ptr(dy), _ptr(dw), _ptr(scratch), N, H, W, C, Co, s, _ptr(w), _ptr(ws), _st())
    _call("cvad_flat_conv3x3_wgrad_staged_bf16", _ptr(act), _ptr(dy), _ptr(dw0), _ptr(scratch), N, H, W, C, Co, s, _st())
    torch.cuda.synchronize()
    assert float(scratch.abs().max()) == 0.0
    assert float((dw - dw0).abs().max()) <= 1e-5 * float(dw0.abs().max())
    wb = w.to(torch.bfloat16).double()
    t = ws[C:2 * C].clone()
    wdw = (wb * dw.double()).sum((0, 2, 3))
    # fp32 partial sums of <= 256 products per block (one block: 256 consecutive weights), fp64 across blocks
    _report(f"{case} T vs sum W*dW", ((t - wdw).abs() / (256 * E * (wb * dw.double()).abs().sum((0, 2, 3)) + 1e-30)).max())
    # ... and that is sum act*dact up to the bf16 rounding of dact (U |dconv|, exact) and the fp32 accumulation of dW, taken here as RUN E
    # relative to |act*dact| (an allowance, not a worst case: the tensor cores sum a CTA's whole pixel range of dW in fp32), 2x slack
    ad = (act.double() * dact.double()).reshape(-1, C)
    _report(f"{case} T vs sum act*dact", ((t - ad.sum(0)).abs() / (2 * (U + RUN * E) * ad.abs().sum(0) + 1e-30)).max())
    del dw, dw0, scratch

    # ---- the one-pass backward against fp64 at the fp32 mean / invstd the kernels received
    draw = torch.full_like(raw, 7.0)
    dg, db = torch.zeros(C, device=dev), torch.zeros(C, device=dev)
    _call("cvad_pad_bn_relu_bwd_tsum_bf16", _ptr(raw), _ptr(dact), _ptr(draw), N, H, W, C, int(phase), _ptr(mean), _ptr(invstd), _ptr(gamma),
          _ptr(beta), _ptr(ws), _ptr(dg), _ptr(db), _st())
    torch.cuda.synchronize()
    assert float(ws.abs().max()) == 0.0, "the workspace is not zero after the backward"
    assert float(draw[:, 0].abs().max()) == 0.0 and float(draw[:, :, -1].abs().max()) == 0.0, "draw border not zero"
    gd = (tc.from_phase(dact, H, W) if phase else tc.from_padded(dact, H, W)).double()
    gb = (tc.from_phase(bits.to(torch.bfloat16), H, W) if phase else tc.from_padded(bits.to(torch.bfloat16), H, W)).double()
    gg = gd * gb
    sh = (1, -1, 1, 1)
    mu, ist, ga, be = mean.double().view(sh), invstd.double().view(sh), gamma.double().view(sh), beta.double().view(sh)
    x = rawf.double()
    xhat = (x - mu) * ist
    S1, S2 = gg.sum((0, 2, 3), keepdim=True), (gg * xhat).sum((0, 2, 3), keepdim=True)
    ref = ist * (ga * gg - ga * S1 / n - xhat * ga * S2 / n)
    got = tc.from_padded(draw, H, W).double()
    # bound per element: bf16 output rounding U |ref|; T differs from gamma*S2 + beta*S1 by <= 2 (U + RUN E) sum |act*dact| (above), which
    # enters as invstd |xhat| / n; the fp32 constants and the fma chain a*g - k0 - k1*x: 8 E over the magnitudes of its three terms
    A = ad.abs().sum(0).view(sh)
    k1 = ist * ist * ga * S2 / n
    bound = U * ref.abs() + ist * xhat.abs() * 2 * (U + RUN * E) * A / n + 8 * E * ((ga * ist * gg).abs() + (ga * ist * S1 / n).abs()
                                                                                  + (k1 * mu).abs() + (k1 * x).abs())
    _report(f"{case} draw", ((got - ref).abs() / bound).max())
    # dgamma / dbeta: fp32 runs of <= RUN terms per thread, fp64 across threads, one fp32 rounding of the result
    gabs, gxabs = gg.abs().sum((0, 2, 3)), (gg * x).abs().sum((0, 2, 3))
    _report(f"{case} dbeta", ((db.double() - S1.flatten()).abs() / (RUN * E * gabs + E * S1.flatten().abs() + 1e-30)).max())
    _report(f"{case} dgamma", ((dg.double() - S2.flatten()).abs() / (RUN * E * invstd.double() * (gxabs + mean.double().abs() * gabs)
                                                                  + E * S2.flatten().abs() + 1e-30)).max())
