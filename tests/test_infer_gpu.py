"""Inference path of the per-frame models (cvad_b200/infer.py): the flat convolution's ReLU-output epilogue against fp64, the frozen bf16
backbone (eval BatchNorm folded into the tensor-core convolutions) against the model's own fp32 backbone, its refresh on weight changes,
and the CUDA-graph streaming scorer against the eager ``ma0.StreamingWindowScorer`` and clip-by-clip scoring.

Every bound is derived from the arithmetic and printed next to the observed error."""
import pytest
import torch
import torch.nn.functional as F

from cvad_b200.noise import DeviceNoise
from test_flat_gpu import FLAT_CASES

pytestmark = pytest.mark.gpu

U32, U16 = 2.0 ** -24, 2.0 ** -8       # unit roundoff of fp32 and bf16


def setup_module(_m):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def rel(a, b, floor=1e-6):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / max(float(b.abs().max()), floor))


def _g(seed):
    return torch.Generator(device="cpu").manual_seed(seed)


def _planes_index(N, Ho, Wo, dev):
    """For the phase planes (4, N, hq, wq) of a padded (N, Ho+2, Wo+2) image: the padded pixel (r, c) each plane position holds
    (plane a*2+b, position (i, j) <- (a + 2i - 2, b + 2j - 2), as tc.to_phase) and whether that pixel exists."""
    hq, wq = (Ho - 1) // 2 + 3, (Wo - 1) // 2 + 3
    a = torch.tensor([0, 0, 1, 1], device=dev).view(4, 1, 1)
    b = torch.tensor([0, 1, 0, 1], device=dev).view(4, 1, 1)
    i = torch.arange(hq, device=dev).view(1, hq, 1)
    j = torch.arange(wq, device=dev).view(1, 1, wq)
    r, c = (a + 2 * i - 2).expand(4, hq, wq), (b + 2 * j - 2).expand(4, hq, wq)
    valid = (r >= 0) & (r <= Ho + 1) & (c >= 0) & (c <= Wo + 1)
    return r.clamp(0, Ho + 1), c.clamp(0, Wo + 1), valid


def _to_planes(padded, Ho, Wo, fill):
    """(N, Ho+2, Wo+2, C) -> (4, N, hq, wq, C); positions without a source pixel get ``fill``."""
    r, c, valid = _planes_index(padded.shape[0], Ho, Wo, padded.device)
    out = padded[:, r, c, :].permute(1, 0, 2, 3, 4)                  # (4, N, hq, wq, C)
    return torch.where(valid.view(4, 1, *valid.shape[1:], 1), out, torch.full_like(out, fill)), valid


# ------------------------------------------------------------------------------------------------ 1. the ReLU-output epilogue
@pytest.mark.parametrize("case", FLAT_CASES)
def test_flat_conv3x3_fwd_relu_vs_fp64(dev, case):
    """cvad_flat_conv3x3_fwd_relu_bf16 after cvad_bn_fold_conv_f32 + pack, both output layouts, against an fp64 conv of the same bf16
    input and the bf16-rounded folded weights, + b', ReLU.

    Bound per element: the kernel sums k = 9*Cin exact bf16 x bf16 products in fp32 and adds b' (k+1 roundings, |err| <= (k+1) U32
    (S + |b'|) with S = sum |x||w'|); the ReLU does not enlarge an error; the bf16 output adds <= U16 |value|.  So
    |y - ref| <= U16 |ref| + (1 + U16) (k+1) U32 (S + |b'|).  Border pixels must be exactly 0; plane positions without a source pixel
    must keep their zero; every other output position starts as NaN."""
    from cvad_b200 import tc
    from cvad_b200.ops import _call, _ptr, _st
    N, H, W, Ci, Co, s = case
    x = torch.randn(N, Ci, H, W, generator=_g(1)).to(dev).to(torch.bfloat16).float()
    w = (torch.randn(Co, Ci, 3, 3, generator=_g(2)) / (3.0 * Ci ** 0.5)).to(dev)
    b = torch.randn(Co, generator=_g(3)).to(dev)
    # BatchNorm of a conv output with sigma ~ 1: gammas of both signs, running means up to 3 sigma off, betas up to 2
    gam = ((torch.rand(Co, generator=_g(4)) + 0.5) * torch.where(torch.rand(Co, generator=_g(5)) < 0.3, -1.0, 1.0)).to(dev)
    beta = ((torch.rand(Co, generator=_g(6)) - 0.5) * 4.0).to(dev)
    rm = ((torch.rand(Co, generator=_g(7)) - 0.5) * 6.0).to(dev)
    rv = (torch.rand(Co, generator=_g(8)) + 0.5).to(dev)
    wf, bf = torch.empty_like(w), torch.empty_like(b)
    _call("cvad_bn_fold_conv_f32", _ptr(w), _ptr(b), _ptr(gam), _ptr(beta), _ptr(rm), _ptr(rv), 1e-5, Co, 9 * Ci, _ptr(wf), _ptr(bf), _st())
    wp = torch.empty(9 * Co, Ci, device=dev, dtype=torch.bfloat16)
    _call("cvad_flat_pack_w3x3_bf16", _ptr(wf), Co, Ci, s, _ptr(wp), None, _st())
    torch.cuda.synchronize()
    wb = wf.to(torch.bfloat16).double()
    pre = F.conv2d(x.double(), wb, bf.double(), stride=s, padding=1)
    S = F.conv2d(x.double().abs(), wb.abs(), bf.double().abs(), stride=s, padding=1)
    del wb
    Ho, Wo = pre.shape[2], pre.shape[3]
    k = 9 * Ci
    ref = torch.zeros(N, Ho + 2, Wo + 2, Co, device=dev, dtype=torch.float64)
    bound = torch.zeros_like(ref)
    ref[:, 1:Ho + 1, 1:Wo + 1] = pre.clamp_min(0).permute(0, 2, 3, 1)
    bound[:, 1:Ho + 1, 1:Wo + 1] = (U16 * pre.clamp_min(0) + (1 + U16) * (k + 1) * U32 * S).permute(0, 2, 3, 1)
    del pre, S
    xin = tc.to_padded(x) if s == 1 else tc.to_phase(x)
    for phase_out in (0, 1):
        if phase_out == 0:
            y = torch.full((N, Ho + 2, Wo + 2, Co), float("nan"), device=dev, dtype=torch.bfloat16)
            want, wbound, valid = ref, bound, None
        else:
            want, valid = _to_planes(ref, Ho, Wo, 0.0)
            wbound, _ = _to_planes(bound, Ho, Wo, 0.0)
            y = torch.where(valid.view(4, 1, *valid.shape[1:], 1), float("nan"), 0.0).expand(-1, N, -1, -1, Co).to(torch.bfloat16).contiguous()
        _call("cvad_flat_conv3x3_fwd_relu_bf16", _ptr(xin), _ptr(wp), _ptr(bf), _ptr(y), N, H, W, Ci, Co, s, phase_out, _st())
        torch.cuda.synchronize()
        err = (y.double() - want).abs()
        ratio = float((err / wbound.clamp_min(1e-300)).nan_to_num(nan=float("inf"))[wbound > 0].max())
        print(f"[relu] {case} phase_out={phase_out}: max |err| / bound = {ratio:.3f}")
        assert not torch.isnan(y).any(), "an output position was left unwritten"
        assert ratio <= 1.0
        assert float(y.double()[wbound == 0].abs().max()) == 0.0, "border pixels / source-less plane positions must be exactly 0"
        if valid is not None:
            assert float(y[:, :, :, :, :].double()[~valid.view(4, 1, *valid.shape[1:], 1).expand_as(y)].abs().max()) == 0.0
        del y, err


def test_flat_conv3x3_fwd_relu_rejects_bad_phase(dev):
    from cvad_b200.ops import _call
    with pytest.raises(RuntimeError, match="cvad_flat_conv3x3_fwd_relu_bf16"):
        _call("cvad_flat_conv3x3_fwd_relu_bf16", None, None, None, None, 1, 8, 8, 32, 32, 1, 2, None)


# ------------------------------------------------------------------------------------------------ 2-3. FrozenBackbone
def _ma_model(dev, seed=4):
    from cvad_b200.ma import CausalAnomalyDetector
    from test_oracle_golden import ma_synth_state
    m = CausalAnomalyDetector()
    m.load_state_dict(ma_synth_state(seed, True), strict=True)
    return m.to(dev).eval()


def _ma0_model(dev, gold):
    """M-A0 with the synthetic state of the golden streaming case (its detector keeps boxes, so the scores follow the features)."""
    from cvad_b200.ma0 import CausalAnomalyDetector
    from test_oracle_golden import ma0_synth_state
    c = [k for k in gold("ma0.pt")["cases"] if k.get("stream")][0]
    m = CausalAnomalyDetector()
    m.load_state_dict(ma0_synth_state(c["seed"], c["margin"]), strict=True)
    return m.to(dev).eval()


class ZeroNoise(DeviceNoise):
    """eps = 0: deterministic under graph replay, so graphed and eager scores can be compared."""

    def normal(self, name, shape, device):
        return torch.zeros(shape, device=device)


# the features of 9 bf16 layers against fp32: every layer rounds its input and its weights to bf16 (<= U16 each, relative); the
# per-layer relative errors add up (the ReLUs and pools do not enlarge them): <= 2 * 9 * U16 relative to the largest feature
FEAT_BOUND = 2 * 9 * U16


@pytest.mark.parametrize("H,W", [(240, 360), (240, 358)])        # stem8 (width % 4 == 0) and the tf32 stem
def test_frozen_backbone_vs_fp32(dev, H, W):
    from cvad_b200 import infer, ops, tc
    m = _ma_model(dev)
    m.noise = ZeroNoise()
    bb = m.backbone
    fz = infer.FrozenBackbone(bb)
    u8 = torch.randint(0, 256, (512, 1, H, W), generator=_g(11), dtype=torch.uint8)
    xf = ((u8.float() - 0.5) / 0.5).to(dev)
    u8 = u8.to(dev)
    f512 = fz(u8)
    # uint8 and host-normalised fp32 frames: bit-identical features
    assert torch.equal(f512, fz(xf))
    # a frame's features do not depend on the batch it came in
    f16 = fz(u8[:16])
    d = float((f16 - f512[:16]).abs().max())
    print(f"[frozen {H}x{W}] batch 16 vs batch 512, max |diff| = {d:.3e}")
    assert d == 0.0
    for n in (16, 512):
        with torch.no_grad():
            bb.precision = "fp32"
            want = bb(xf[:n].unsqueeze(0))[0]
            bb.precision = "bf16"
        e = rel(f512[:n], want)
        print(f"[frozen {H}x{W}] N={n}: features rel err {e:.2e} (bound {FEAT_BOUND:.2e})")
        assert e <= FEAT_BOUND
        with torch.no_grad():
            got_s = m.tail(f512[:n].view(-1, 16, f512.shape[1]))["anomaly_scores"]
            want_s = m.tail(want.view(-1, 16, want.shape[1]))["anomaly_scores"]
        es = rel(got_s, want_s)
        print(f"[frozen {H}x{W}] N={n}: scores rel err {es:.2e} (tolerance 1e-3)")
        assert es < 1e-3 and torch.equal(got_s > 0.5, want_s > 0.5)
    if (H, W) == (240, 360):
        x = u8[:16]
        fz(x)
        n0 = ops.LAUNCHES[0]
        fz(x)
        n_frozen = ops.LAUNCHES[0] - n0
        n0 = ops.LAUNCHES[0]
        with torch.no_grad():
            tc.backbone_forward_bf16(bb, x)
        n_eval = ops.LAUNCHES[0] - n0
        print(f"[frozen] ABI calls per backbone call: FrozenBackbone {n_frozen}, eval _BackboneBF16 {n_eval}")
        assert n_frozen == 11 and n_eval == 36


# ------------------------------------------------------------------------------------------------ 4-5. refresh and the graphed scorer
def _score_clip_by_clip(m, seq, T, stride, n_win):
    """Each window as its own clip through a fresh FrozenBackbone + model.tail."""
    from cvad_b200 import infer
    fz = infer.FrozenBackbone(m.backbone)
    out = []
    with torch.no_grad():
        for w in range(n_win):
            f = fz(seq[w * stride: w * stride + T])
            out.append(m.tail(f.unsqueeze(0))["anomaly_scores"])
    return torch.cat(out)


def test_frozen_backbone_refresh(dev):
    """In-place weight / running-statistic changes and load_state_dict are picked up; the result equals a fresh snapshot bit for bit."""
    from cvad_b200 import infer
    from test_oracle_golden import ma_synth_state
    m = _ma_model(dev)
    bb = m.backbone
    x = torch.randint(0, 256, (16, 1, 64, 96), generator=_g(12), dtype=torch.uint8).to(dev)
    fz = infer.FrozenBackbone(bb)
    f0 = fz(x)
    bufs = [t.data_ptr() for f in fz.folded for t in f]
    with torch.no_grad():
        bb.layer2[0].weight.mul_(1.25)
        bb.layer3[4].running_var.mul_(1.5)
    f1 = fz(x)
    assert not torch.equal(f0, f1)
    assert torch.equal(f1, infer.FrozenBackbone(bb)(x))
    m.load_state_dict(ma_synth_state(5, True), strict=True)
    f2 = fz(x)
    assert torch.equal(f2, infer.FrozenBackbone(bb)(x))
    assert bufs == [t.data_ptr() for f in fz.folded for t in f], "in-place refresh must re-fold into the same buffers"
    # a replaced tensor drops the snapshot
    bb.layer1[0].weight = torch.nn.Parameter(bb.layer1[0].weight.detach() * 0.5)
    f3 = fz(x)
    assert torch.equal(f3, infer.FrozenBackbone(bb)(x)) and not torch.equal(f3, f2)


CHUNKS = (5, 8, 3, 7, 1, 4, 8, 8, 4, 4, 2)        # 54 frames: pushes completing no window, repeated sizes; capacity 24 wraps


@pytest.mark.parametrize("kind", ["ma", "ma0"])
def test_graphed_streaming_scorer(dev, gold, kind):
    from cvad_b200 import infer
    from cvad_b200.ma0 import StreamingWindowScorer
    m = _ma_model(dev) if kind == "ma" else _ma0_model(dev, gold)
    m.noise = ZeroNoise()
    T, stride, cap, H, W = 16, 4, 24, 64, 96
    seq = torch.randint(0, 256, (sum(CHUNKS), 1, H, W), generator=_g(13), dtype=torch.uint8).to(dev)
    m.set_precision("bf16")
    gs = infer.GraphedStreamingScorer(m, clip_len=T, stride=stride, capacity=cap)
    es = StreamingWindowScorer(m, clip_len=T, stride=stride, capacity=cap)
    ref_fz = infer.FrozenBackbone(m.backbone)
    ring_ref = torch.zeros(cap, 6144, device=dev)
    got, pos, keys = [], 0, set()
    for n in CHUNKS:
        chunk = seq[pos:pos + n]
        s, w0 = gs.push(chunk)
        se, we0 = es.push(chunk)
        assert w0 == we0 and s.shape == se.shape, (n, w0, we0, s.shape, se.shape)
        with torch.no_grad():
            f = ref_fz(chunk)
        for r in range(n):
            ring_ref[(pos + r) % cap] = f[r]
        pos += n
        keys.add((n, s.shape[0]))
        # the ring and the cursor hold exactly what the pushes wrote: capturing (and its warm-up runs) did not advance the stream
        assert torch.equal(gs.ring, ring_ref)
        assert gs.cursor.tolist() == [pos, w0 + s.shape[0]] == [gs.n_frames, gs.next_window]
        got.append(s)
    got = torch.cat(got)
    n_win = (pos - T) // stride + 1
    assert got.shape[0] == n_win and len(gs.graphs) == len(keys), (len(gs.graphs), keys)
    want = _score_clip_by_clip(m, seq, T, stride, n_win)
    e = rel(got, want)
    with torch.no_grad():
        m.set_precision("fp32")
        clips = torch.stack([seq[w * stride: w * stride + T] for w in range(n_win)])
        want32 = m(clips)["anomaly_scores"]
        m.set_precision("bf16")
    e32 = rel(got, want32)
    print(f"[graphed {kind}] {n_win} windows, {len(gs.graphs)} graphs: vs FrozenBackbone clip by clip {e:.2e} (2e-5), vs fp32 {e32:.2e} (1e-3)")
    assert e < 2e-5 and e32 < 1e-3


def test_graphed_scorer_follows_weight_updates(dev):
    """In-place updates (an optimizer step, load_state_dict) reach the captured graphs; a replaced tensor makes the scorer capture again.
    A frame's features enter the ring when it is pushed, with the weights of that moment (as in ma0.StreamingWindowScorer), so after each
    change four pushes of 4 frames fill one window with frames that all arrived after it; that window is checked: its ring rows bit for
    bit against a fresh FrozenBackbone, its score against clip-by-clip scoring."""
    from cvad_b200 import infer
    from test_oracle_golden import ma_synth_state
    m = _ma_model(dev)
    m.noise = ZeroNoise()
    T, stride, cap = 16, 4, 24
    seq = torch.randint(0, 256, (16 + 3 * 16, 1, 64, 96), generator=_g(14), dtype=torch.uint8).to(dev)
    gs = infer.GraphedStreamingScorer(m, clip_len=T, stride=stride, capacity=cap)
    gs.push(seq[:8])
    gs.push(seq[8:16])
    assert len(gs.graphs) == 2

    def four_pushes(p0):
        for p in range(p0, p0 + 16, 4):
            s, w0 = gs.push(seq[p:p + 4])
        fz = infer.FrozenBackbone(m.backbone)
        for p in range(p0, p0 + 16, 4):
            f = fz(seq[p:p + 4])
            for r in range(4):
                assert torch.equal(gs.ring[(p + r) % cap], f[r]), (p0, p + r)
        want = _score_clip_by_clip(m, seq, T, stride, w0 + 1)[w0:]
        assert w0 * stride == p0 and rel(s, want) < 2e-5, (p0, s, want)
    with torch.no_grad():
        m.backbone.layer2[0].weight.mul_(1.25)
        m.backbone.layer3[4].running_var.mul_(1.5)
    four_pushes(16)
    assert len(gs.graphs) == 3
    m.load_state_dict(ma_synth_state(5, True), strict=True)
    four_pushes(32)
    assert len(gs.graphs) == 3
    m.backbone.layer1[0].weight = torch.nn.Parameter(m.backbone.layer1[0].weight.detach() * 0.5)
    four_pushes(48)
    assert len(gs.graphs) == 1          # dropped and captured again


def test_graphed_scorer_errors_match_eager(dev):
    from cvad_b200 import infer
    from cvad_b200.ma0 import StreamingWindowScorer
    m = _ma_model(dev)
    m.train()
    for cls in (StreamingWindowScorer, infer.GraphedStreamingScorer):
        with pytest.raises(RuntimeError, match=r"needs model\.eval\(\)"):
            cls(m)
    m.eval()
    msgs = []
    for cls in (StreamingWindowScorer, infer.GraphedStreamingScorer):
        sc = cls(m, clip_len=16, stride=4, capacity=24)
        got = []
        for bad in (torch.zeros(9, 1, 64, 96, dtype=torch.uint8, device=dev), torch.zeros(4, 1, 64, 96, dtype=torch.uint8),
                    torch.zeros(1, 64, 96, dtype=torch.uint8, device=dev)):
            with pytest.raises((RuntimeError, ValueError)) as ei:
                sc.push(bad)
            got.append((type(ei.value), str(ei.value)))
        msgs.append(got)
        with pytest.raises(ValueError, match="ring capacity"):
            cls(m, clip_len=16, stride=4, capacity=19)
    assert msgs[0] == msgs[1], msgs
