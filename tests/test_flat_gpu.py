"""Parity of the flat (TMA + tcgen05) backbone kernels on the B200 against plain PyTorch fp32 ops on the same bf16-rounded
operands: convolution forward / data-gradient / weight-gradient for stride 1 and 2, and the padded-layout BN / pool /
stem kernels in both activation layouts (padded-flat and phase planes)."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def setup_module(_m):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def rel(a, b, floor=1e-6):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / max(float(b.abs().max()), floor))


def _g(seed):
    return torch.Generator(device="cpu").manual_seed(seed)


# N, H, W, Cin, Cout, stride -- the reference's eight layer shapes (cad:150-153) at small / ragged frame counts, plus one
# case large enough for several 512-row tiles per CTA
FLAT_CASES = [(3, 12, 17, 32, 32, 1), (2, 9, 11, 64, 64, 1), (2, 8, 12, 128, 128, 1), (1, 8, 12, 256, 256, 1),
              (2, 12, 18, 32, 64, 2), (3, 15, 23, 64, 128, 2), (2, 15, 23, 128, 256, 2), (1, 7, 9, 32, 32, 1),
              (40, 60, 90, 32, 32, 1), (24, 30, 45, 64, 64, 1), (9, 60, 90, 32, 64, 2)]
# the seven distinct layer shapes of the BENCHMARKED step (512 frames of 240x360, cad:150-153): every template instance bench.py
# launches gets here the same number of work items per CTA (2-3 for Cin >= 128, 10-19 for the 32/64-channel layers), so accumulator-
# ring wrap-around, weight-ring parity across items and the multi-CTA weight-gradient grids are checked where the benchmark runs them
FLAT_CASES += [(512, 60, 90, 32, 32, 1), (512, 60, 90, 32, 64, 2), (512, 30, 45, 64, 64, 1), (512, 30, 45, 64, 128, 2),
               (512, 15, 23, 128, 128, 1), (512, 15, 23, 128, 256, 2), (512, 8, 12, 256, 256, 1)]


def _inputs(dev, N, H, W, Ci, Co, s):
    x = torch.randn(N, Ci, H, W, generator=_g(1)).to(dev).to(torch.bfloat16).float()
    w = (torch.randn(Co, Ci, 3, 3, generator=_g(2)) / (3.0 * Ci ** 0.5)).to(dev)
    b = torch.randn(Co, generator=_g(3)).to(dev)
    xr = x.clone().requires_grad_(True)
    wr = w.to(torch.bfloat16).float().requires_grad_(True)
    ref = F.conv2d(xr, wr, b, stride=s, padding=1)
    dy = torch.randn(ref.shape, generator=_g(4)).to(dev).to(torch.bfloat16).float()
    gx, gw = torch.autograd.grad(ref, (xr, wr), dy)
    return x, w, b, ref.detach(), dy, gx, gw


@pytest.mark.parametrize("case", FLAT_CASES)
def test_flat_conv3x3_fwd_fused_bn_statistics(dev, case):
    """cvad_flat_conv3x3_fwd_stats_bf16: same output as the plain forward, and the epilogue's per-channel sum / sum of squares over the
    interior pixels equal those of the bf16 output it wrote (what the separate statistics pass would read back)."""
    from cvad_b200 import tc
    from cvad_b200.ops import _call, _ptr, _st
    N, H, W, Ci, Co, s = case
    x, w, b, ref, _, _, _ = _inputs(dev, *case)
    Ho, Wo = ref.shape[2], ref.shape[3]
    wf = torch.empty(9 * Co, Ci, device=dev, dtype=torch.bfloat16)
    _call("cvad_flat_pack_w3x3_bf16", _ptr(w), Co, Ci, s, _ptr(wf), None, _st())
    xin = tc.to_padded(x) if s == 1 else tc.to_phase(x)
    y0 = torch.full((N, Ho + 2, Wo + 2, Co), 7.0, device=dev, dtype=torch.bfloat16)
    y1 = torch.full_like(y0, 7.0)
    _call("cvad_flat_conv3x3_fwd_bf16", _ptr(xin), _ptr(wf), _ptr(b), _ptr(y0), N, H, W, Ci, Co, s, _st())
    ws = torch.zeros(2 * Co, device=dev, dtype=torch.float64)
    _call("cvad_flat_conv3x3_fwd_stats_bf16", _ptr(xin), _ptr(wf), _ptr(b), _ptr(y1), N, H, W, Ci, Co, s, _ptr(ws), _st())
    torch.cuda.synchronize()
    assert torch.equal(tc.from_padded(y0, Ho, Wo), tc.from_padded(y1, Ho, Wo))
    inner = y1[:, 1:Ho + 1, 1:Wo + 1, :].double()
    s1, s2 = inner.sum(dim=(0, 1, 2)), (inner * inner).sum(dim=(0, 1, 2))
    assert rel(ws[:Co], s1, floor=1.0) < 2e-5 and rel(ws[Co:], s2) < 2e-5
    # finalize -> mean / invstd / running statistics as nn.BatchNorm2d computes them from that tensor; ws comes back zeroed
    mean, invstd = torch.empty(Co, device=dev), torch.empty(Co, device=dev)
    rm, rv, nbt = torch.zeros(Co, device=dev), torch.ones(Co, device=dev), torch.tensor(0, device=dev)
    cnt = N * Ho * Wo
    _call("cvad_bn_finalize_f64", _ptr(ws), Co, float(cnt), 1e-5, 0.1, _ptr(mean), _ptr(invstd), _ptr(rm), _ptr(rv), _ptr(nbt), _st())
    torch.cuda.synchronize()
    flat = inner.reshape(-1, Co)
    var = flat.var(dim=0, unbiased=False)
    assert rel(mean.double(), flat.mean(dim=0), floor=1e-2) < 1e-4 and rel(invstd.double(), (var + 1e-5).rsqrt()) < 1e-4
    assert rel(rv.double(), 0.9 + 0.1 * flat.var(dim=0, unbiased=True)) < 1e-4 and int(nbt) == 1
    assert float(ws.abs().max()) == 0.0


@pytest.mark.parametrize("case", FLAT_CASES)
def test_flat_conv3x3_fwd_dgrad_wgrad(dev, case):
    from cvad_b200 import tc
    from cvad_b200.ops import _call, _ptr, _st
    N, H, W, Ci, Co, s = case
    x, w, b, ref, dy, gx, gw = _inputs(dev, *case)
    Ho, Wo = ref.shape[2], ref.shape[3]
    wf = torch.empty(9 * Co, Ci, device=dev, dtype=torch.bfloat16)
    wd = torch.empty(9 * Ci, Co, device=dev, dtype=torch.bfloat16)
    _call("cvad_flat_pack_w3x3_bf16", _ptr(w), Co, Ci, s, _ptr(wf), _ptr(wd), _st())
    xin = tc.to_padded(x) if s == 1 else tc.to_phase(x)
    # junk-filled outputs: the kernels must write every interior element themselves
    y = torch.full((N, Ho + 2, Wo + 2, Co), 7.0, device=dev, dtype=torch.bfloat16)
    _call("cvad_flat_conv3x3_fwd_bf16", _ptr(xin), _ptr(wf), _ptr(b), _ptr(y), N, H, W, Ci, Co, s, _st())
    torch.cuda.synchronize()
    e_f = rel(tc.from_padded(y, Ho, Wo), ref)
    dyp = tc.to_padded(dy)
    dx = torch.full(xin.shape, 7.0, device=dev, dtype=torch.bfloat16)
    _call("cvad_flat_conv3x3_dgrad_bf16", _ptr(dyp), _ptr(wd), _ptr(dx), N, H, W, Ci, Co, s, _st())
    torch.cuda.synchronize()
    dxr = tc.from_padded(dx, H, W) if s == 1 else tc.from_phase(dx, H, W)
    e_d = rel(dxr, gx)
    dw = torch.zeros(Co, Ci, 3, 3, device=dev)
    _call("cvad_flat_conv3x3_wgrad_bf16", _ptr(xin), _ptr(dyp), _ptr(dw), N, H, W, Ci, Co, s, _st())
    torch.cuda.synchronize()
    e_w = rel(dw, gw)
    # staged variant: accumulates on top of what dw already holds and hands the staging buffer back zeroed
    dw2 = dw.clone()
    scratch = torch.zeros(9 * Co * Ci, device=dev)
    _call("cvad_flat_conv3x3_wgrad_staged_bf16", _ptr(xin), _ptr(dyp), _ptr(dw2), _ptr(scratch), N, H, W, Ci, Co, s, _st())
    torch.cuda.synchronize()
    e_w2 = rel(dw2, 2 * gw)
    assert float(scratch.abs().max()) == 0.0
    print(f"[flat] {case}: fwd {e_f:.2e} dgrad {e_d:.2e} wgrad {e_w:.2e} staged {e_w2:.2e}")
    assert e_f < 1e-2 and e_d < 1e-2 and e_w < 2e-3 and e_w2 < 2e-3


@pytest.mark.parametrize("case", FLAT_CASES)
def test_flat_dgrad_fused_bn_backward_reductions(dev, case):
    """cvad_flat_conv3x3_dgrad_bnstats_bf16: the same dx as the plain data-gradient, and its epilogue's per-channel sums
    sum g / sum g*xhat (g = dx * [bn(raw) > 0] over the interior pixels, from the bf16 dx it stored) equal what the BatchNorm
    backward's own reduce pass computes from raw and dx -- for padded-flat (stride 1) and phase-plane (stride 2) outputs."""
    from cvad_b200 import tc
    from cvad_b200.ops import _call, _ptr, _st
    N, H, W, Ci, Co, s = case
    x, w, b, ref, dy, gx, gw = _inputs(dev, *case)
    wd = torch.empty(9 * Ci, Co, device=dev, dtype=torch.bfloat16)
    _call("cvad_flat_pack_w3x3_bf16", _ptr(w), Co, Ci, s, None, _ptr(wd), _st())
    dyp = tc.to_padded(dy)
    shape = (N, H + 2, W + 2, Ci) if s == 1 else tuple(tc.act_shape(N, H, W, Ci, True))
    dx0 = torch.full(shape, 7.0, device=dev, dtype=torch.bfloat16)
    dx1 = torch.full(shape, 7.0, device=dev, dtype=torch.bfloat16)
    _call("cvad_flat_conv3x3_dgrad_bf16", _ptr(dyp), _ptr(wd), _ptr(dx0), N, H, W, Ci, Co, s, _st())
    # the layer below: raw (junk border), BatchNorm scale / shift chosen so that roughly half of the ReLUs are open
    rawf = (torch.randn(N, Ci, H, W, generator=_g(21)) * 1.5 + 0.3).to(dev).to(torch.bfloat16).float()
    raw = tc.to_padded(rawf)
    raw[:, 0] = 9.0
    raw[:, :, -1] = -5.0
    gam = (torch.rand(Ci, generator=_g(22)) + 0.5).to(dev)
    gam[::5] *= -1.0
    bet = (torch.randn(Ci, generator=_g(23)) * 0.3).to(dev)
    mean = (torch.randn(Ci, generator=_g(24)) * 0.2 + 0.3).to(dev)
    invstd = (torch.rand(Ci, generator=_g(25)) * 0.5 + 0.4).to(dev)
    ws = torch.zeros(2 * Ci, device=dev, dtype=torch.float64)
    _call("cvad_flat_conv3x3_dgrad_bnstats_bf16", _ptr(dyp), _ptr(wd), _ptr(dx1), N, H, W, Ci, Co, s, _ptr(raw), _ptr(gam), _ptr(bet), _ptr(mean),
          _ptr(invstd), _ptr(ws), _st())
    torch.cuda.synchronize()
    d0 = tc.from_padded(dx0, H, W) if s == 1 else tc.from_phase(dx0, H, W)
    d1 = tc.from_padded(dx1, H, W) if s == 1 else tc.from_phase(dx1, H, W)
    assert torch.equal(d0, d1)
    sh = (1, -1, 1, 1)
    ga = (gam * invstd).view(sh)
    gate = (rawf * ga + (bet.view(sh) - mean.view(sh) * ga)) > 0
    g = (d1 * gate).double()
    xhat = ((rawf - mean.view(sh)) * invstd.view(sh)).double()
    s0, s1 = g.sum(dim=(0, 2, 3)), (g * xhat).sum(dim=(0, 2, 3))
    scale = float(g.abs().sum(dim=(0, 2, 3)).max())
    e0, e1 = float((ws[:Ci] - s0).abs().max()) / scale, float((ws[Ci:] - s1).abs().max()) / scale
    print(f"[flat] {case}: fused BN-backward sums, error relative to sum|g|: {e0:.2e} / {e1:.2e}")
    assert e0 < 2e-5 and e1 < 5e-5


def test_layout_helpers_roundtrip(dev):
    from cvad_b200 import tc
    x = torch.randn(2, 8, 15, 23, generator=_g(1)).to(dev).to(torch.bfloat16).float()
    assert torch.equal(tc.from_padded(tc.to_padded(x), 15, 23), x)
    assert torch.equal(tc.from_phase(tc.to_phase(x), 15, 23), x)
    x = torch.randn(1, 8, 60, 90, generator=_g(2)).to(dev).to(torch.bfloat16).float()
    assert torch.equal(tc.from_phase(tc.to_phase(x), 60, 90), x)


@pytest.mark.parametrize("C,H,W,phase", [(32, 12, 18, 0), (32, 12, 18, 1), (64, 15, 23, 1), (128, 15, 23, 0), (256, 8, 12, 0), (64, 9, 7, 1)])
@pytest.mark.parametrize("training", [True, False])
def test_pad_bn_relu_fwd_bwd(dev, C, H, W, phase, training):
    """stats + apply (+ phase-plane output) and the fused ReLU+BN backward (dact given in the same layout as act)."""
    from cvad_b200 import ops, tc
    from cvad_b200.ops import _call, _ptr, _st
    N = 3
    x = (torch.randn(N, C, H, W, generator=_g(1)) * 2 + 1).to(dev).to(torch.bfloat16).float()
    raw = tc.to_padded(x)
    raw[:, 0] = 9.0                      # convolution outputs carry junk in their border
    raw[:, :, 0] = -9.0
    raw[:, -1] = 5.0
    raw[:, :, -1] = 3.0
    xr = x.clone().requires_grad_(True)
    gam = (torch.rand(C, generator=_g(2)) + 0.5).to(dev).requires_grad_(True)
    bet = torch.randn(C, generator=_g(3)).to(dev).requires_grad_(True)
    rm = (torch.randn(C, generator=_g(12)) * 0.1 + 1).to(dev)
    rv = (torch.rand(C, generator=_g(13)) + 3.5).to(dev)
    rm2, rv2 = rm.clone(), rv.clone()
    ref = F.relu(F.batch_norm(xr, rm, rv, gam, bet, training, 0.1, 1e-5))
    mean, invstd = torch.empty(C, device=dev), torch.empty(C, device=dev)
    nbt = torch.tensor(0, device=dev)
    if training:
        _call("cvad_pad_bn_stats_bf16", _ptr(raw), N, H, W, C, _ptr(ops.bn_workspace(dev, C)), 1e-5, 0.1, _ptr(mean), _ptr(invstd), _ptr(rm2),
              _ptr(rv2), _ptr(nbt), _st())
        assert rel(rm2, rm) < 1e-4 and rel(rv2, rv) < 1e-4 and int(nbt) == 1
    else:
        _call("cvad_bn_eval_prepare_f32", C, 1e-5, _ptr(rm2), _ptr(rv2), _ptr(mean), _ptr(invstd), _st())
    act = torch.full(tc.act_shape(N, H, W, C, phase), 7.0, device=dev, dtype=torch.bfloat16)
    _call("cvad_pad_bn_apply_relu_bf16", _ptr(raw), _ptr(act), N, H, W, C, phase, _ptr(mean), _ptr(invstd), _ptr(gam), _ptr(bet), _st())
    torch.cuda.synchronize()
    expect = tc.to_phase(ref.detach()) if phase else tc.to_padded(ref.detach())
    assert rel(act.float(), expect.float()) < 1e-2
    ones = torch.ones(N, C, H, W, device=dev)
    hole = (tc.to_phase(ones) if phase else tc.to_padded(ones)) == 0
    assert float(act[hole].float().abs().max()) == 0.0      # exact zeros wherever no pixel maps (conv padding)
    g = torch.randn(N, C, H, W, generator=_g(5)).to(dev).to(torch.bfloat16).float()
    dact = tc.to_phase(g) if phase else tc.to_padded(g)
    if not phase:
        dact[:, 0] = 11.0                # data-gradients carry junk in their border as well
        dact[:, :, -1] = -4.0
    gr = torch.autograd.grad(ref, (xr, gam, bet), g)
    draw = torch.full(raw.shape, 7.0, device=dev, dtype=torch.bfloat16)
    dg, db = torch.zeros(C, device=dev), torch.zeros(C, device=dev)
    _call("cvad_pad_bn_relu_bwd_bf16", _ptr(raw), _ptr(dact), _ptr(draw), N, H, W, C, phase, _ptr(mean), _ptr(invstd), _ptr(gam), _ptr(bet),
          int(training), _ptr(ops.bn_workspace(dev, C)), _ptr(dg), _ptr(db), _st())
    torch.cuda.synchronize()
    assert rel(tc.from_padded(draw, H, W), gr[0]) < 1e-2
    border = draw.clone()
    border[:, 1:H + 1, 1:W + 1] = 0
    assert float(border.float().abs().max()) == 0.0
    assert rel(dg, gr[1]) < 2e-3 and rel(db, gr[2]) < 2e-3


# 9x14 -> 4x6 has overlapping bins of unequal size; 8x12 (the benchmarked step's last layer) and 12x18 divide evenly, so the per-frame
# backward takes its uniform-bin branch
AVGPOOL_CASES = [(3, 64, 9, 14), (512, 256, 8, 12), (2, 32, 12, 18)]


def test_pad_avgpool(dev):
    from cvad_b200 import tc
    from cvad_b200.ops import _call, _ptr, _st
    for N, C, H, W in AVGPOOL_CASES:
        x = torch.randn(N, C, H, W, generator=_g(1)).to(dev).to(torch.bfloat16).float()
        xp = tc.to_padded(x)
        xp[:, 0] = 5.0
        feats = torch.empty(N, C, 4, 6, device=dev)
        _call("cvad_pad_avgpool_bf16_fwd", _ptr(xp), N, H, W, C, 4, 6, _ptr(feats), _st())
        xr = x.clone().requires_grad_(True)
        pr = F.adaptive_avg_pool2d(xr, (4, 6))
        e_f = rel(feats, pr.detach())
        go = torch.randn(N, C, 4, 6, generator=_g(6)).to(dev)
        (gxr,) = torch.autograd.grad(pr, xr, go)
        dxp = torch.zeros(N, H + 2, W + 2, C, device=dev, dtype=torch.bfloat16)
        dxp[:, 1:H + 1, 1:W + 1] = float("nan")          # every interior element must be written
        _call("cvad_pad_avgpool_bf16_bwd", _ptr(go), N, H, W, C, 4, 6, _ptr(dxp), _st())
        e_b = rel(tc.from_padded(dxp, H, W), gxr)
        print(f"[avgpool] {(N, C, H, W)}: fwd {e_f:.2e} bwd {e_b:.2e}")
        assert e_f < 1e-5, (N, C, H, W, e_f)
        assert e_b < 1e-2, (N, C, H, W, e_b)        # a NaN left in dx fails here as well


# frame shapes of the tf32 stem -> status of its fused pass 2 + max-pool: 801 (cudaErrorNotSupported) where a band of 7 convolution rows
# needs more 128-position sub-tiles than the 16-slot accumulator ring holds (602 px wide: 17), and the unfused pair is the only path
STEM_TF32_FUSED_STATUS = {(2, 37, 53): 0, (3, 240, 360): 0, (1, 16, 20): 0, (5, 64, 64): 0, (40, 240, 360): 0, (2, 50, 36): 0,
                          (1, 20, 602): 801}


@pytest.mark.parametrize("N,H,W", list(STEM_TF32_FUSED_STATUS))
@pytest.mark.parametrize("training", [True, False])
def test_stem_tf32(dev, N, H, W, training):
    """conv 7x7 s2 p3 1->32 + bn1 (+ running statistics) + relu + maxpool(3,2,1), tf32 tensor-core passes vs fp32 torch."""
    from cvad_b200 import ops, tc
    from cvad_b200.ops import _call, _ptr, _st
    x = (torch.rand(N, 1, H, W, generator=_g(1)) * 255.0).round().sub(0.5).div(0.5).to(dev)     # the reference's [-1, 509] range
    w = (torch.randn(32, 1, 7, 7, generator=_g(2)) * 0.1).to(dev)
    b = torch.randn(32, generator=_g(3)).to(dev)
    gam = (torch.rand(32, generator=_g(4)) + 0.5).to(dev)
    bet = torch.randn(32, generator=_g(5)).to(dev)
    rm = torch.randn(32, generator=_g(6)).to(dev)
    rv = (torch.rand(32, generator=_g(7)) * 100 + 50).to(dev)
    rm2, rv2 = rm.clone(), rv.clone()
    y = F.conv2d(x, w, b, stride=2, padding=3)
    ref = F.max_pool2d(F.relu(F.batch_norm(y, rm, rv, gam, bet, training, 0.1, 1e-5)), 3, 2, 1)
    mean, invstd = torch.empty(32, device=dev), torch.empty(32, device=dev)
    nbt = torch.tensor(0, device=dev)
    x_nchw = x
    x = torch.full((int(ops.L().cvad_stem_x4_floats(N, H, W)),), float("nan"), device=dev)      # 2x2 space-to-depth buffer
    _call("cvad_stem_space_to_depth_f32", _ptr(x_nchw), N, H, W, _ptr(x), _st())
    if training:
        _call("cvad_stem_tf32_stats", _ptr(x), _ptr(w), _ptr(b), N, H, W, _ptr(ops.bn_workspace(dev, 32)), 1e-5, 0.1, _ptr(mean), _ptr(invstd),
              _ptr(rm2), _ptr(rv2), _ptr(nbt), _st())
        assert rel(rm2, rm) < 1e-3 and rel(rv2, rv) < 2e-3 and int(nbt) == 1
    else:
        _call("cvad_bn_eval_prepare_f32", 32, 1e-5, _ptr(rm2), _ptr(rv2), _ptr(mean), _ptr(invstd), _st())
    Ho, Wo = y.shape[2], y.shape[3]
    y1 = torch.full((N, Ho, Wo, 32), 7.0, device=dev, dtype=torch.bfloat16)
    _call("cvad_stem_tf32_bn_relu", _ptr(x), _ptr(w), _ptr(b), N, H, W, _ptr(mean), _ptr(invstd), _ptr(gam), _ptr(bet), _ptr(y1), _st())
    PH, PW = ref.shape[2], ref.shape[3]
    a0 = torch.full((N, PH + 2, PW + 2, 32), 7.0, device=dev, dtype=torch.bfloat16)
    _call("cvad_pad_maxpool3x3s2_bf16", _ptr(y1), N, Ho, Wo, 32, _ptr(a0), _st())
    torch.cuda.synchronize()
    e = rel(a0.float(), tc.to_padded(ref).float())
    print(f"[stem] N={N} {H}x{W} training={training}: rel err {e:.2e}")
    assert e < 1e-2
    # pass 2 + max-pool as ONE kernel (bands pooled out of shared memory): bit-identical to the two kernels, zero border included
    a1 = torch.full((N, PH + 2, PW + 2, 32), 7.0, device=dev, dtype=torch.bfloat16)
    status = _call("cvad_stem_tf32_bn_relu_maxpool", _ptr(x), _ptr(w), _ptr(b), N, H, W, _ptr(mean), _ptr(invstd), _ptr(gam), _ptr(bet), _ptr(a1), _st(),
                   accept=(801,))
    torch.cuda.synchronize()
    assert status == STEM_TF32_FUSED_STATUS[(N, H, W)]
    if status == 0:
        assert torch.equal(a0, a1)
    else:
        assert bool((a1 == 7.0).all())                                   # a declined call writes nothing


@pytest.mark.parametrize("u8", [False, True])
def test_stem_forward_wide_frame_falls_back(dev, u8):
    """tc.stem_forward on a frame too wide for both fused stems (W not a multiple of 4, a band does not fit) takes the unfused tf32
    pass 2 and the separate max-pool: bit-identical to calling that pair directly, from fp32 and from uint8 frames."""
    import types
    from cvad_b200 import ops, tc
    from cvad_b200.ops import _call, _ptr, _st
    N, H, W = 1, 20, 602
    raw = (torch.rand(N, 1, H, W, generator=_g(1)) * 255.0).round()
    x = raw.sub(0.5).div(0.5).to(dev)
    bb = types.SimpleNamespace(conv1=torch.nn.Conv2d(1, 32, 7, 2, 3).to(dev), bn1=torch.nn.BatchNorm2d(32).to(dev), input_mean=0.5,
                               input_std=0.5)
    with torch.no_grad():
        bb.conv1.weight.copy_(torch.randn(32, 1, 7, 7, generator=_g(2)) * 0.1)
        bb.conv1.bias.copy_(torch.randn(32, generator=_g(3)))
        bb.bn1.weight.copy_(torch.rand(32, generator=_g(4)) + 0.5)
        bb.bn1.bias.copy_(torch.randn(32, generator=_g(5)))
    mean, invstd = torch.randn(32, generator=_g(6)).to(dev), (torch.rand(32, generator=_g(7)) + 0.5).to(dev)
    assert int(ops.L().cvad_stem8_bytes(N, H, W)) == -1
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    PH, PW = (Ho - 1) // 2 + 1, (Wo - 1) // 2 + 1
    x4 = torch.empty(int(ops.L().cvad_stem_x4_floats(N, H, W)), device=dev)
    _call("cvad_stem_space_to_depth_f32", _ptr(x), N, H, W, _ptr(x4), _st())
    y1 = torch.empty(N, Ho, Wo, 32, device=dev, dtype=torch.bfloat16)
    _call("cvad_stem_tf32_bn_relu", _ptr(x4), _ptr(bb.conv1.weight), _ptr(bb.conv1.bias), N, H, W, _ptr(mean), _ptr(invstd),
          _ptr(bb.bn1.weight), _ptr(bb.bn1.bias), _ptr(y1), _st())
    ref = torch.full((N, PH + 2, PW + 2, 32), 7.0, device=dev, dtype=torch.bfloat16)
    _call("cvad_pad_maxpool3x3s2_bf16", _ptr(y1), N, Ho, Wo, 32, _ptr(ref), _st())
    a = torch.full_like(ref, 7.0)
    tc.stem_forward(bb, raw.to(torch.uint8).to(dev) if u8 else x, a, mean, invstd)
    torch.cuda.synchronize()
    assert torch.equal(a, ref)


@pytest.mark.parametrize("N,H,W", [(2, 37, 52), (3, 240, 360), (1, 16, 20), (5, 64, 64), (40, 240, 360), (2, 50, 36), (2, 120, 180)])
@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("u8", [False, True])
def test_stem_f16_space_to_depth_2x4(dev, N, H, W, training, u8):
    """The stem's fp16 formulation (kind::f16 over a 2x4 space-to-depth, N = 64 = (output parity, channel), pass 2 fused with the max-pool)
    vs fp32 torch: conv 7x7 s2 p3 1->32 + bn1 (+ running statistics) + relu + maxpool(3,2,1), from fp32 and from uint8 frames."""
    from cvad_b200 import ops, tc
    from cvad_b200.ops import _call, _ptr, _st
    raw = (torch.rand(N, 1, H, W, generator=_g(1)) * 255.0).round()
    x = raw.sub(0.5).div(0.5).to(dev)                                   # the reference's [-1, 509] range
    w = (torch.randn(32, 1, 7, 7, generator=_g(2)) * 0.1).to(dev)
    b = torch.randn(32, generator=_g(3)).to(dev)
    gam = (torch.rand(32, generator=_g(4)) + 0.5).to(dev)
    bet = torch.randn(32, generator=_g(5)).to(dev)
    rm = torch.randn(32, generator=_g(6)).to(dev)
    rv = (torch.rand(32, generator=_g(7)) * 100 + 50).to(dev)
    rm2, rv2 = rm.clone(), rv.clone()
    y = F.conv2d(x, w, b, stride=2, padding=3)
    ref = F.max_pool2d(F.relu(F.batch_norm(y, rm, rv, gam, bet, training, 0.1, 1e-5)), 3, 2, 1)
    nb = int(ops.L().cvad_stem8_bytes(N, H, W))
    assert nb > 0
    x8 = torch.full((nb,), 0x7e, device=dev, dtype=torch.uint8)        # fp16 NaN pattern: every pixel must be written
    if u8:
        _call("cvad_stem8_space_to_depth_u8", _ptr(raw.to(torch.uint8).to(dev)), N, H, W, 0.5, 0.5, _ptr(x8), _st())
    else:
        _call("cvad_stem8_space_to_depth_f32", _ptr(x), N, H, W, _ptr(x8), _st())
    mean, invstd = torch.empty(32, device=dev), torch.empty(32, device=dev)
    nbt = torch.tensor(0, device=dev)
    if training:
        _call("cvad_stem8_f16_stats", _ptr(x8), _ptr(w), _ptr(b), N, H, W, _ptr(ops.bn_workspace(dev, 32)), 1e-5, 0.1, _ptr(mean), _ptr(invstd),
              _ptr(rm2), _ptr(rv2), _ptr(nbt), _st())
        assert rel(rm2, rm) < 1e-3 and rel(rv2, rv) < 2e-3 and int(nbt) == 1
    else:
        _call("cvad_bn_eval_prepare_f32", 32, 1e-5, _ptr(rm2), _ptr(rv2), _ptr(mean), _ptr(invstd), _st())
    PH, PW = ref.shape[2], ref.shape[3]
    a1 = torch.full((N, PH + 2, PW + 2, 32), 7.0, device=dev, dtype=torch.bfloat16)
    _call("cvad_stem8_f16_bn_relu_maxpool", _ptr(x8), _ptr(w), _ptr(b), N, H, W, _ptr(mean), _ptr(invstd), _ptr(gam), _ptr(bet), _ptr(a1), _st())
    torch.cuda.synchronize()
    e = rel(a1.float(), tc.to_padded(ref).float())
    print(f"[stem f16] N={N} {H}x{W} training={training} u8={u8}: rel err {e:.2e}")
    assert e < 1e-2
    border = a1.clone()
    border[:, 1:-1, 1:-1] = 0
    assert float(border.float().abs().max()) == 0.0                      # the zero border of the padded-flat output


def test_stem_f16_declines_other_widths(dev):
    from cvad_b200 import ops
    assert int(ops.L().cvad_stem8_bytes(2, 37, 53)) == -1 and int(ops.L().cvad_stem8_bytes(2, 37, 54)) == -1
