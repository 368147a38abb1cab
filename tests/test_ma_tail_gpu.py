"""M-A's causal branch (csrc/ma_tail.cu through ma_ops.py) against a float64 reference.

Part A calls every entry point of ma_tail.cu on fp32 inputs with its outputs pre-filled with NaN / sentinels, and compares with a float64
restatement on the same fp32 inputs (oracle/ma.py where it has one); backward references come from float64 autograd.  Part B runs the
whole branch through ``model.tail()`` at the benchmarked shape (B = 32, T = 16) with a detector head engineered so that the batch holds
every track count, fallback frames beside real detections, compaction gaps and tracks that come and go, and compares values and every
tail gradient elementwise with ``oracle.ma.ma_tail`` in float64.

Three kinds of bound:
* gathers, masks and copies are exact;
* short sums and pointwise math are held to a few fp32 unit roundoffs of the sum of the absolute terms, derived next to each check;
* the GRU and the composed branch are held to a yardstick measured in the test: the error of the same fp32 computation run by torch on
  the CPU against float64.  In the composed branch the yardstick takes the two 6144-wide projections from the project's tensor-core GEMM
  (whose accumulation is not IEEE fp32; it has tests of its own), so the bound measures what the rest of the branch adds.  The kernel's
  error must be <= 4 x the yardstick plus 64 fp32 ulps of the tensor's scale.
Every check prints its observed error-to-bound ratio.
"""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

U = 2.0 ** -24                    # fp32 unit roundoff: |fl(v) - v| <= U |v|
MAXDET, NF, HID = 5, 6, 64
NODE = 32                         # the structure learner's node width (pair rows are 2 x 32 wide)
SCALE = (360.0, 240.0, 80.0, 120.0)
OFF = (0.0, 0.0, 15.0, 25.0)
LO = (10.0, 10.0, 10.0, 20.0)
HI = (350.0, 230.0, 100.0, 150.0)
MARGIN_PX = 1e-2                  # every box coordinate stays this far from the validity window's edges (fp32 and fp64 agree on validity)
GRID_CAP_THREADS = 8 * 148 * 128  # the grid-stride launches cap at 8 CTAs of 128 threads per SM (148 SMs on a B200)


def _call(name, *args):
    """One ABI entry; tensor arguments are passed as pointers.  They stay referenced until the launch is enqueued: a pointer taken from
    a temporary (``x.to(dev)``) would be handed back to the caching allocator, and to the next input, before the kernel runs."""
    from cvad_b200.ops import _call as call
    call(name, *[a.data_ptr() if isinstance(a, torch.Tensor) else a for a in args])


def _st():
    return torch.cuda.current_stream().cuda_stream


def nan_like(shape, dev, dtype=torch.float32):
    return torch.full(shape, float("nan"), device=dev, dtype=dtype)


def sentinel_i32(shape, dev):
    return torch.full(shape, -7, device=dev, dtype=torch.int32)


def check(name, got, ref, bound):
    """|got - ref| <= bound elementwise (bound 0 = exact); got must be finite.  Returns the worst error / bound."""
    got, ref, bound = (torch.as_tensor(v).double().cpu() for v in (got, ref, bound))
    bound = bound.expand_as(ref)
    assert torch.isfinite(got).all(), f"{name}: non-finite (unwritten) output"
    err = (got - ref).abs()
    exact = bound == 0
    assert torch.equal(got[exact], ref[exact]), f"{name}: exact slots differ"
    ratio = float((err[~exact] / bound[~exact]).max()) if (~exact).any() else 0.0
    print(f"[ma_tail] {name}: err/bound {ratio:.3f}")
    assert ratio <= 1.0, (name, ratio)
    return ratio


def ulp32(scale):
    return float(np.spacing(np.float32(max(scale, 1e-30))))


def check_yard(name, got, ref, cpu32, mask=None):
    """Kernel error <= 4 x (torch-CPU fp32 error) + 64 fp32 ulps of the tensor's scale, both against float64."""
    got, ref, cpu32 = (torch.as_tensor(v).double().cpu() for v in (got, ref, cpu32))
    if mask is not None:
        got, ref, cpu32 = got[mask], ref[mask], cpu32[mask]
    assert torch.isfinite(got).all(), f"{name}: non-finite output"
    err = float((got - ref).abs().max()) if got.numel() else 0.0
    yard = float((cpu32 - ref).abs().max()) if got.numel() else 0.0
    scale = float(ref.abs().max()) if got.numel() else 0.0
    bound = 4.0 * yard + 64.0 * ulp32(scale)
    ratio = err / bound if bound > 0 else (0.0 if err == 0 else math.inf)
    print(f"[ma_tail] {name}: err {err:.3e} yardstick {yard:.3e} scale {scale:.3e} err/bound {ratio:.3f}")
    assert ratio <= 1.0, (name, err, yard, scale)
    return ratio


def _logit(p):
    return math.log(p / (1.0 - p))


# ================================================================================================ part A: entry points
def _det_raw(R, gen):
    """raw (R,5,4) fp32 and the intended validity (R,5): frame r uses subset r % 32 of the anchors.  Valid anchors have x, y inside the
    window; an invalid one has x or y outside it, rotating over both coordinates and both sides.  (w = 80 s + 15 and h = 120 s + 25 lie
    strictly inside their windows for every logit, so only x and y can invalidate an anchor.)  Coordinates stay >= 1e-2 px from the
    window edges; some logits are saturated (|raw| = 30)."""
    raw = torch.empty(R, MAXDET, 4, dtype=torch.float64)
    valid = torch.zeros(R, MAXDET, dtype=torch.bool)
    u = lambda a, b: a + (b - a) * float(torch.rand((), generator=gen, dtype=torch.float64))
    rot = 0
    for r in range(R):
        mask = r % 32
        for k in range(MAXDET):
            ok = bool(mask >> k & 1)
            valid[r, k] = ok
            for c in range(4):
                lo, hi = _logit((LO[c] - OFF[c]) / SCALE[c]) if c < 2 else -30.0, _logit((HI[c] - OFF[c]) / SCALE[c]) if c < 2 else 30.0
                raw[r, k, c] = u(lo + 0.05, hi - 0.05) if c < 2 else (30.0 if (r + k + c) % 7 == 0 else -30.0 if (r + k + c) % 7 == 1 else u(-8, 8))
            if not ok:
                c, side = rot % 2, rot // 2 % 2
                rot += 1
                lo, hi = _logit((LO[c] - OFF[c]) / SCALE[c]), _logit((HI[c] - OFF[c]) / SCALE[c])
                raw[r, k, c] = (30.0 if rot % 3 == 0 else u(hi + 0.05, 25.0)) if side else (-30.0 if rot % 3 == 0 else u(-25.0, lo - 0.05))
    return raw.float(), valid


def _box64(raw):
    s = torch.sigmoid(raw.double())
    return s * torch.tensor(SCALE, dtype=torch.float64) + torch.tensor(OFF, dtype=torch.float64), s


def test_det_decode_fwd_bwd(dev):
    """Every validity subset of the 5 anchors (counts 0..5, every compaction pattern), saturated logits, the fallback box, the flag."""
    gen = torch.Generator().manual_seed(101)
    R = 4 * 32
    raw, valid = _det_raw(R, gen)
    box64, s64 = _box64(raw)
    lo, hi = torch.tensor(LO, dtype=torch.float64), torch.tensor(HI, dtype=torch.float64)
    assert torch.equal(((box64 >= lo) & (box64 <= hi)).all(-1), valid)
    assert float(torch.minimum((box64 - lo).abs(), (box64 - hi).abs()).min()) >= MARGIN_PX      # fp32 and fp64 agree on validity
    rd = raw.to(dev)
    box, cnt, src = nan_like((R, MAXDET, 4), dev), sentinel_i32((R,), dev), sentinel_i32((R, MAXDET), dev)
    flag = torch.full((1,), 0.5, device=dev)
    _call("cvad_det_decode_f32", rd, R, box, cnt, src, flag, _st())
    # reference: in-order compaction of the valid anchors, fallback row when none survives
    want_cnt = valid.sum(1).clamp(min=1)
    want_src = torch.full((R, MAXDET), -1, dtype=torch.int64)
    want_box = torch.zeros(R, MAXDET, 4, dtype=torch.float64)
    exact = torch.ones(R, MAXDET, 4, dtype=torch.bool)
    for r in range(R):
        ks = valid[r].nonzero().flatten()
        want_src[r, :len(ks)] = ks
        if len(ks):
            want_box[r, :len(ks)] = box64[r, ks]
            exact[r, :len(ks)] = False
        else:
            want_box[r, 0] = torch.tensor([180.0, 120.0, 30.0, 60.0])
    assert torch.equal(cnt.cpu().long(), want_cnt)
    assert torch.equal(src.cpu().long(), want_src)
    assert float(flag) == 1.0
    # box = fl(fl(sigmoid) * scale + off): sigmoid = 1 / (1 + expf(-v)) carries <= 2 ulp (4U) from expf, U from the add and U from the
    # division (6U relative); the product and the add round once each: <= 8U (s scale + off)
    terms = torch.zeros_like(want_box)
    for r in range(R):
        ks = valid[r].nonzero().flatten()
        terms[r, :len(ks)] = s64[r, ks] * torch.tensor(SCALE, dtype=torch.float64) + torch.tensor(OFF, dtype=torch.float64)
    check("det_decode box", box, want_box, torch.where(exact, torch.zeros_like(terms), 8 * U * terms))
    # backward: draw[src[k]] = dbox[k] * scale * s (1 - s); 0 for every anchor that was not kept
    dbox = torch.randn(R, MAXDET, 4, generator=gen)
    draw = nan_like((R, MAXDET, 4), dev)
    _call("cvad_det_decode_bwd_f32", rd, dbox.to(dev), src, R, draw, _st())
    want = torch.zeros(R, MAXDET, 4, dtype=torch.float64)
    bound = torch.zeros_like(want)
    sc = torch.tensor(SCALE, dtype=torch.float64)
    for r in range(R):
        for k, j in enumerate(valid[r].nonzero().flatten().tolist()):
            want[r, j] = dbox[r, k].double() * sc * s64[r, j] * (1 - s64[r, j])
            # s carries 6U relative, so 1 - s carries <= 7U s absolute (cancellation near s = 1); the three products add 3U relative:
            # |err| <= |dbox| scale s (7U + 9U (1 - s)) <= 16U |dbox| scale s
            bound[r, j] = 16 * U * dbox[r, k].double().abs() * sc * s64[r, j]
    check("det_decode_bwd draw", draw, want, bound)
    assert (draw.cpu()[~valid] == 0).all()
    # a batch in which every frame falls back leaves the flag at its prior value
    raw0 = torch.full((6, MAXDET, 4), -30.0, device=dev)
    box0, cnt0, src0 = nan_like((6, MAXDET, 4), dev), sentinel_i32((6,), dev), sentinel_i32((6, MAXDET), dev)
    flag0 = torch.full((1,), 0.25, device=dev)
    _call("cvad_det_decode_f32", raw0, 6, box0, cnt0, src0, flag0, _st())
    assert float(flag0) == 0.25 and (cnt0.cpu() == 1).all() and (src0.cpu() == -1).all()
    assert torch.equal(box0.cpu()[:, 0], torch.tensor([180.0, 120.0, 30.0, 60.0]).expand(6, 4))
    assert (box0.cpu()[:, 1:] == 0).all()


@pytest.mark.parametrize("B,T,D", [(7, 16, 64), (5, 1, 64), (6, 3, 5)])
def test_traj_assemble_fwd_bwd(dev, B, T, D):
    """Counts vary over a clip's frames, every track count 1..5 appears; traj / dbox / dreid are gathers and must be bit-identical."""
    gen = torch.Generator().manual_seed(200 + T)
    ntr_want = torch.tensor([1 + b % 5 for b in range(B)])
    cnt = torch.stack([torch.randint(1, int(n) + 1, (T,), generator=gen) for n in ntr_want])
    cnt[torch.arange(B), torch.randint(0, T, (B,), generator=gen)] = ntr_want        # the clip's maximum is reached in some frame
    box, reid = torch.randn(B, T, MAXDET, 4, generator=gen), torch.randn(B, T, MAXDET, D, generator=gen)
    traj, ntr = nan_like((B, MAXDET, T, 4 + D), dev), sentinel_i32((B,), dev)
    flag = torch.full((1,), 0.5, device=dev)
    c32 = cnt.to(torch.int32).to(dev)
    _call("cvad_traj_assemble_f32", box.to(dev), reid.to(dev), c32, B, T, D, traj, ntr, flag, _st())
    ok = (torch.arange(MAXDET).view(1, 1, -1) < cnt.unsqueeze(-1)).unsqueeze(-1).float()
    want = (torch.cat([box, reid], -1) * ok).permute(0, 2, 1, 3)
    assert torch.equal(ntr.cpu().long(), cnt.max(1).values) and torch.equal(ntr.cpu().long(), ntr_want)
    assert torch.equal(traj.cpu(), want)
    assert float(flag) == (1.0 if int(ntr_want.max()) >= 2 else 0.5)
    dtraj = torch.randn(B, MAXDET, T, 4 + D, generator=gen)
    dbox, dreid = nan_like((B, T, MAXDET, 4), dev), nan_like((B, T, MAXDET, D), dev)
    _call("cvad_traj_assemble_bwd_f32", dtraj.to(dev), c32, B, T, D, dbox, dreid, _st())
    g = dtraj.permute(0, 2, 1, 3) * ok
    assert torch.equal(dbox.cpu(), g[..., :4]) and torch.equal(dreid.cpu(), g[..., 4:])
    # every clip with one track: the flag keeps its prior value
    one = torch.ones(B, T, dtype=torch.int32, device=dev)
    flag1 = torch.full((1,), 0.25, device=dev)
    _call("cvad_traj_assemble_f32", box.to(dev), reid.to(dev), one, B, T, D, traj, ntr, flag1, _st())
    assert float(flag1) == 0.25 and (ntr.cpu() == 1).all()


def _gru_ref(gi, w, b, mask, dhT):
    """oracle.ma.gru_last on gi itself (W_ih = I, b_ih = 0 makes its input projection the identity) and its autograd gradients,
    in gi's dtype; dhT is applied to the active tracks only."""
    from oracle.ma import gru_last
    dt = gi.dtype
    gi, w, b = (v.detach().to(dt).clone().requires_grad_(True) for v in (gi, w, b))
    P = {"traj_encoder.gru.weight_ih_l0": torch.eye(3 * HID, dtype=dt), "traj_encoder.gru.bias_ih_l0": torch.zeros(3 * HID, dtype=dt),
         "traj_encoder.gru.weight_hh_l0": w, "traj_encoder.gru.bias_hh_l0": b}
    hT = gru_last(P, gi)
    (hT * (dhT.to(dt) * mask.view(-1, 1))).sum().backward()
    return hT.detach(), gi.grad, w.grad, b.grad


@pytest.mark.parametrize("B,T,sat", [(1, 1, False), (3, 4, False), (32, 16, False), (7, 64, False), (32, 16, True)])
def test_gru_fwd_bwd(dev, B, T, sat):
    """hT, dgi, dW_hh, db_hh against the fp64 recurrence; inactive tracks exactly 0; the inference path is bit-identical to the
    training path; a second backward accumulates into .grad."""
    from cvad_b200 import ma_ops
    gen = torch.Generator().manual_seed(300 + 7 * B + T + sat)
    N = B * MAXDET
    ntr = torch.tensor([1 + (b * 3) % 5 for b in range(B)], dtype=torch.int32)
    mask = (torch.arange(MAXDET).view(1, -1) < ntr.view(-1, 1).long()).flatten()
    gi = torch.randn(N, T, 3 * HID, generator=gen) * (6.0 if sat else 0.7)
    w = (torch.rand(3 * HID, HID, generator=gen) * 2 - 1) / 8 * (4.0 if sat else 1.0)
    b = (torch.rand(3 * HID, generator=gen) * 2 - 1) / 8
    dhT = torch.randn(N, HID, generator=gen)
    h64, dgi64, dw64, db64 = _gru_ref(gi.double(), w, b, mask.double(), dhT)
    h32, dgi32, dw32, db32 = _gru_ref(gi, w, b, mask.float(), dhT)
    gd, wd, bd, nd = gi.to(dev), w.to(dev), b.to(dev), ntr.to(dev)
    hT, saved = nan_like((N, HID), dev), nan_like((N, T, 5, HID), dev)
    _call("cvad_gru_fwd_f32", gd, wd, bd, nd, B, T, hT, saved, _st())
    hT_inf = nan_like((N, HID), dev)
    _call("cvad_gru_fwd_f32", gd, wd, bd, nd, B, T, hT_inf, None, _st())
    assert torch.equal(hT_inf, hT)
    assert (hT.cpu()[~mask] == 0).all()
    check_yard(f"gru hT B{B} T{T}{' sat' if sat else ''}", hT.cpu()[mask], h64[mask], h32[mask])
    dgi, dw, db = nan_like((N, T, 3 * HID), dev), torch.zeros(3 * HID, HID, device=dev), torch.zeros(3 * HID, device=dev)
    _call("cvad_gru_bwd_f32", dhT.to(dev), saved, wd, nd, B, T, dgi, dw, db, _st())
    assert (dgi.cpu()[~mask] == 0).all()
    check_yard(f"gru dgi B{B} T{T}{' sat' if sat else ''}", dgi, dgi64, dgi32)
    check_yard(f"gru dW_hh B{B} T{T}{' sat' if sat else ''}", dw, dw64, dw32)
    check_yard(f"gru db_hh B{B} T{T}{' sat' if sat else ''}", db, db64, db32)
    # through the autograd wrapper: W_hh / b_hh gradients accumulate into .grad (the arena semantics), dgi is returned
    gl = gd.clone().requires_grad_(True)
    wp, bp = torch.nn.Parameter(wd.clone()), torch.nn.Parameter(bd.clone())
    for rep in (1, 2):
        h = ma_ops.gru_last(gl, wp, bp, nd)
        h.backward(dhT.to(dev))
        assert torch.equal(h.detach(), hT)
        check_yard(f"gru wrapper dW_hh x{rep}", wp.grad, rep * dw64, rep * dw32)
        check_yard(f"gru wrapper db_hh x{rep}", bp.grad, rep * db64, rep * db32)
    check_yard("gru wrapper dgi x2", gl.grad, 2 * dgi64, 2 * dgi32)


@pytest.mark.parametrize("B", [5, 300])
def test_reparam_kl_fwd_bwd(dev, B):
    gen = torch.Generator().manual_seed(400 + B)
    ntr = torch.tensor([1 + b % 5 for b in range(B)], dtype=torch.int32)
    act = (torch.arange(MAXDET).view(1, -1, 1) < ntr.view(-1, 1, 1).long()).expand(B, MAXDET, NF)
    mu = torch.randn(B, MAXDET, NF, generator=gen) * 2
    lv = torch.rand(B, MAXDET, NF, generator=gen) * 16 - 8
    lv[0, 0, :2] = torch.tensor([-8.0, 8.0])
    eps = torch.randn(B, MAXDET, NF, generator=gen)
    dz, dkl = torch.randn(B, MAXDET, NF, generator=gen), torch.randn(B, generator=gen)
    z, kl = nan_like((B, MAXDET, NF), dev), nan_like((B,), dev)
    args = [t.to(dev) for t in (mu, lv, eps, ntr)]
    _call("cvad_reparam_kl_f32", *args, B, z, kl, _st())
    m, l, e = (v.double().requires_grad_(True) for v in (mu, lv, eps))
    z64 = (m + e * torch.exp(0.5 * l)) * act
    terms = -0.5 * (1 + l - m * m - l.exp()) * act
    kl64 = terms.sum((1, 2)) / ntr.double()
    (z64 * dz.double()).sum().add((kl64 * dkl.double()).sum()).backward()
    md, ld, ed, n = mu.double(), lv.double(), eps.double(), ntr.double()
    zero = ~act
    # z = fl(m + fl(eps fl(expf(0.5 l)))): expf <= 4U, the product and the sum U each: <= 6U (|m| + |eps e^{l/2}|)
    zb = 6 * U * (md.abs() + (ed * torch.exp(0.5 * ld)).abs())
    check("reparam z", z, z64.detach(), torch.where(zero, torch.zeros_like(zb), zb))
    # kl: each term is a 4-term sum with expf (<= 8U of its absolute terms), 30 terms are summed by a 5-level shuffle tree (5U) and
    # divided by nt (U): <= 16U sum|terms| / nt
    kb = 16 * U * (0.5 * (1 + ld.abs() + md * md + ld.exp()) * act).sum((1, 2)) / n
    check("reparam kl", kl, kl64.detach(), kb)
    dmu, dlv = nan_like((B, MAXDET, NF), dev), nan_like((B, MAXDET, NF), dev)
    _call("cvad_reparam_kl_bwd_f32", *args, B, dz.to(dev), dkl.to(dev), dmu, dlv, _st())
    gk = (dkl.double() / n).view(-1, 1, 1)
    # dmu = g + gk m: <= 4U (|g| + |gk m|); dlv = g eps 0.5 e^{l/2} - 0.5 gk (1 - e^l): expf 4U, 3 products, 2 adds: <= 10U sum|terms|
    b_mu = 4 * U * (dz.double().abs() + (gk * md).abs())
    b_lv = 10 * U * ((dz.double() * ed * 0.5 * torch.exp(0.5 * ld)).abs() + (gk.abs() * 0.5 * (1 + ld.exp())))
    check("reparam_bwd dmu", dmu, m.grad, torch.where(zero, torch.zeros_like(b_mu), b_mu))
    check("reparam_bwd dlogvar", dlv, l.grad, torch.where(zero, torch.zeros_like(b_lv), b_lv))


def _ntr(B, gen):
    return torch.randint(1, MAXDET + 1, (B,), generator=gen, dtype=torch.int32)


@pytest.mark.parametrize("B", [1, 32, 300, 5000])
@pytest.mark.parametrize("Hn", [NODE, 7])
def test_pair_concat_fwd_bwd(dev, B, Hn):
    """Bit-exact forward; the backward sums 10 terms.  B = 300 and 5000 at the model's width wrap the grid-stride loop."""
    if B >= 300 and Hn == NODE:
        assert B * 25 * 2 * Hn > GRID_CAP_THREADS
    gen = torch.Generator().manual_seed(500 + B + Hn)
    node = torch.randn(B, MAXDET, Hn, generator=gen)
    pair = nan_like((B, MAXDET, MAXDET, 2 * Hn), dev)
    _call("cvad_pair_concat_f32", node.to(dev), B, Hn, pair, _st())
    want = torch.cat([node.unsqueeze(2).expand(B, MAXDET, MAXDET, Hn), node.unsqueeze(1).expand(B, MAXDET, MAXDET, Hn)], -1)
    assert torch.equal(pair.cpu(), want)
    dpair = torch.randn(B, MAXDET, MAXDET, 2 * Hn, generator=gen)
    dnode = nan_like((B, MAXDET, Hn), dev)
    _call("cvad_pair_concat_bwd_f32", dpair.to(dev), B, Hn, dnode, _st())
    d = dpair.double()
    ref = d[..., :Hn].sum(2) + d[..., Hn:].sum(1)
    absum = d[..., :Hn].abs().sum(2) + d[..., Hn:].abs().sum(1)
    check(f"pair_concat_bwd B{B} Hn{Hn}", dnode, ref, 10 * U * absum)        # recursive 10-term sum: <= 9U sum|terms|


@pytest.mark.parametrize("B", [1, 32, 300, 5000])
def test_adj_structured_fwd_bwd(dev, B):
    """adj_assemble both directions bit-exact (zero diagonal, zero row / column 5, zeros at i or j >= ntr); structured and its backward
    are 5- and 6-term fma sums.  B = 5000 wraps the grid-stride loops."""
    gen = torch.Generator().manual_seed(600 + B)
    ntr = _ntr(B, gen)
    ntr[: min(B, 5)] = torch.arange(1, min(B, 5) + 1, dtype=torch.int32)
    e = torch.rand(B, MAXDET, MAXDET, generator=gen)
    adj = nan_like((B, NF, NF), dev)
    nd = ntr.to(dev)
    _call("cvad_adj_assemble_f32", e.to(dev), nd, B, adj, 0, _st())
    ok = (torch.arange(MAXDET).view(1, -1) < ntr.view(-1, 1).long()).float()
    emask = ok.unsqueeze(2) * ok.unsqueeze(1) * (1 - torch.eye(MAXDET))
    want = torch.zeros(B, NF, NF)
    want[:, :MAXDET, :MAXDET] = e * emask
    assert torch.equal(adj.cpu(), want)
    dadj = torch.randn(B, NF, NF, generator=gen)
    de = nan_like((B, MAXDET, MAXDET), dev)
    _call("cvad_adj_assemble_f32", dadj.to(dev), nd, B, de, 1, _st())
    assert torch.equal(de.cpu(), dadj[:, :MAXDET, :MAXDET] * emask)
    # structured[b,k,i] = sum_j adj[b,i,j] z[b,k,j] on a dense adjacency (every entry exercised)
    a = torch.randn(B, NF, NF, generator=gen)
    z = torch.randn(B, MAXDET, NF, generator=gen)
    out = nan_like((B, MAXDET, NF), dev)
    ad, zd = a.to(dev), z.to(dev)
    _call("cvad_structured_f32", ad, zd, B, out, _st())
    a64, z64 = a.double().requires_grad_(True), z.double().requires_grad_(True)
    s64 = torch.einsum("bij,bkj->bki", a64, z64)
    check(f"structured B{B}", out, s64.detach(), 6 * U * torch.einsum("bij,bkj->bki", a64.abs(), z64.abs()).detach())
    dout = torch.randn(B, MAXDET, NF, generator=gen)
    (s64 * dout.double()).sum().backward()
    g_adj, g_z = nan_like((B, NF, NF), dev), nan_like((B, MAXDET, NF), dev)
    _call("cvad_structured_bwd_f32", ad, zd, dout.to(dev), B, g_adj, g_z, _st())
    do = dout.double().abs()
    check(f"structured_bwd dadj B{B}", g_adj, a64.grad, 5 * U * torch.einsum("bki,bkj->bij", do, z.double().abs()))
    check(f"structured_bwd dz B{B}", g_z, z64.grad, 6 * U * torch.einsum("bki,bij->bkj", do, a.double().abs()))


@pytest.mark.parametrize("B", [5, 32, 300, 5000])
def test_scorer_inputs_fwd_bwd(dev, B):
    """Masked means over every track count; factors with cur == pred exactly take the zero subgradient of |.|, as torch does."""
    gen = torch.Generator().manual_seed(700 + B)
    ntr = _ntr(B, gen)
    ntr[: min(B, 5)] = torch.arange(1, min(B, 5) + 1, dtype=torch.int32)
    z = torch.randn(B, MAXDET, NF, generator=gen)
    pred = torch.randn(B, MAXDET, NF, generator=gen)
    pred[:, :, 0] = z[:, :, 0]                   # factor 0: identical sums in the same order, so cur == pred exactly
    pred[::3, :, 4] = z[::3, :, 4]
    cin, mn, tin = nan_like((B, 18), dev), nan_like((B, 12), dev), nan_like((B, 6), dev)
    nd = ntr.to(dev)
    _call("cvad_scorer_inputs_f32", z.to(dev), pred.to(dev), nd, B, cin, mn, tin, _st())
    ok = (torch.arange(MAXDET).view(1, -1, 1) < ntr.view(-1, 1, 1).long()).double()
    n = ntr.double().view(-1, 1)
    cur, prd = (z.double() * ok).sum(1) / n, (pred.double() * ok).sum(1) / n
    tied = cur == prd
    assert tied[:, 0].all() and not tied[:, 1:4].any()
    # mean of nt terms: (nt - 1)U sum|z| / nt from the sum, U from the division: <= 6U sum|z| / nt
    bc, bp = 6 * U * (z.double().abs() * ok).sum(1) / n, 6 * U * (pred.double().abs() * ok).sum(1) / n
    cur, prd = cur.detach(), prd.detach()
    assert ((cur - prd).abs() > bc + bp)[~tied].all()                  # the sign of cur - prd is the same in fp32
    check(f"scorer_inputs cin B{B}", cin, torch.cat([cur, prd, (cur - prd).abs()], -1), torch.cat([bc, bp, bc + bp + U * (cur.abs() + prd.abs())], -1))
    check(f"scorer_inputs min B{B}", mn, torch.cat([cur, prd], -1), torch.cat([bc, bp], -1))
    check(f"scorer_inputs tin B{B}", tin, cur, bc)
    assert (cin.cpu()[:, 12][tied[:, 0]] == 0).all()
    dcin, dmn, dtin = torch.randn(B, 18, generator=gen), torch.randn(B, 12, generator=gen), torch.randn(B, 6, generator=gen)
    dz, dp = nan_like((B, MAXDET, NF), dev), nan_like((B, MAXDET, NF), dev)
    _call("cvad_scorer_inputs_bwd_f32", cin, nd, B, dcin.to(dev), dmn.to(dev), dtin.to(dev), dz, dp, _st())
    # reference on the kernel's own (fp32) cur / prd, as the backward consumes them
    c32 = cin.cpu().double()
    cur2, prd2 = c32[:, :6].clone().requires_grad_(True), c32[:, 6:12].clone().requires_grad_(True)
    (torch.cat([cur2, prd2, (cur2 - prd2).abs()], -1) * dcin.double()).sum().add(
        (torch.cat([cur2, prd2], -1) * dmn.double()).sum()).add((cur2 * dtin.double()).sum()).backward()
    gz, gp = (cur2.grad.unsqueeze(1) / n.unsqueeze(1)) * ok, (prd2.grad.unsqueeze(1) / n.unsqueeze(1)) * ok
    # gc = 4-term sum, gp = 3-term sum, then / nt: <= 4U sum|terms| / nt
    sc = (dcin.double()[:, :6].abs() + dmn.double()[:, :6].abs() + dtin.double().abs() + dcin.double()[:, 12:].abs()) / n
    sp = (dcin.double()[:, 6:12].abs() + dmn.double()[:, 6:].abs() + dcin.double()[:, 12:].abs()) / n
    check(f"scorer_inputs_bwd dz B{B}", dz, gz, 4 * U * sc.unsqueeze(1) * ok)
    check(f"scorer_inputs_bwd dpred B{B}", dp, gp, 4 * U * sp.unsqueeze(1) * ok)


@pytest.mark.parametrize("n", [1, 1001, 2 * GRID_CAP_THREADS + 3])
def test_lincomb3(dev, n):
    gen = torch.Generator().manual_seed(800 + n % 97)
    x, y, z = (torch.randn(n, generator=gen) for _ in range(3))
    a, b, c = 0.5, -0.3, 0.2
    out = nan_like((n,), dev)
    _call("cvad_lincomb3_f32", out, x.to(dev), a, y.to(dev), b, z.to(dev), c, n, _st())
    af, bf, cf = (float(np.float32(v)) for v in (a, b, c))     # the coefficients as the kernel receives them
    terms = (af * x.double()).abs() + (bf * y.double()).abs() + (cf * z.double()).abs()
    # three products and two adds (fma-contracted or not): <= 4U sum|terms|
    check(f"lincomb3 n{n}", out, af * x.double() + bf * y.double() + cf * z.double(), 4 * U * terms)


@pytest.mark.parametrize("C", [1, 2, 7, 64])
def test_softmax_rows_fwd_bwd(dev, C):
    gen = torch.Generator().manual_seed(900 + C)
    rows = 1000 if C == 64 else GRID_CAP_THREADS + 77            # past the grid-stride cap for the narrow rows
    x = torch.randn(rows, C, generator=gen) * 4
    x[0] = 80.0
    x[1, :] = -80.0
    if C > 1:
        x[2, 0], x[3, C - 1] = 80.0, -80.0
        x[4] = torch.where(torch.arange(C) % 2 == 0, 80.0, -80.0)
    y = nan_like((rows, C), dev)
    _call("cvad_softmax_rows_f32", x.to(dev), rows, C, y, _st())
    xd = x.double()
    y64 = torch.softmax(xd, -1)
    dm = (xd - xd.max(-1, keepdim=True).values).abs()
    # e_c = expf(x_c - m): the subtraction perturbs the exponent by U|x_c - m|, expf adds 4U; s sums C such terms ((C - 1)U); the
    # division adds U:  |err y_c| <= U y_c (|x_c - m| + sum_j y_j |x_j - m| + C + 10).  An e_c below fp32's normal range (the -80 logits
    # beside +80) loses its relative precision or flushes to 0: with s >= 1 that costs at most 2^-126 absolute.
    bound = U * y64 * (dm + (y64 * dm).sum(-1, keepdim=True) + C + 10) + 2.0 ** -126
    check(f"softmax_rows C{C}", y, y64, bound)
    dy = torch.randn(rows, C, generator=gen)
    dx = nan_like((rows, C), dev)
    _call("cvad_softmax_rows_bwd_f32", y, dy.to(dev), rows, C, dx, _st())
    yk, dyd = y.cpu().double(), dy.double()                      # reference on the kernel's own y, as the backward consumes it
    dot = (yk * dyd).sum(-1, keepdim=True)
    ref = yk * (dyd - dot)
    # dot: C-term sum of products (C U sum|y dy|); dx = y (dy - dot): two roundings of |y (dy - dot)|, or 2^-150 each where that product
    # is subnormal (the y of a -80 logit)
    bwd = 2 * U * (yk * (dyd - dot)).abs() + yk * (C + 1) * U * (yk * dyd).abs().sum(-1, keepdim=True) + 2.0 ** -149
    check(f"softmax_rows_bwd C{C}", dx, ref, bwd)


# ================================================================================================ part B: model.tail() at B = 32, T = 16
BB, TT, FEAT = 32, 16, 6144
KINK_MARGIN = 1e-5                  # relative distance of every detector / classifier ReLU input from 0 (vs the sum of its |terms|)
ANCHOR_ORDER = (3, 1, 4, 0, 2)      # the order in which anchors become valid as the score rises: every count below 5 has a gap


def _keep(train):
    import synth
    if not train:
        return {}
    return {"det0": synth.keep_mask((BB, TT, 512), 0.3, 1002), "det1": synth.keep_mask((BB, TT, 256), 0.2, 1003),
            "scorer0": synth.keep_mask((BB, 64), 0.2, 1004), "cls0": synth.keep_mask((BB, 512), 0.3, 1005),
            "cls1": synth.keep_mask((BB, 256), 0.2, 1006)}


def _engineer_head(P, feats, keep, train, mode):
    """Last detector layer for a chosen detection pattern.  One score per frame, s = u . h8 (h8 the 64-wide input of the last layer,
    in fp64), decides everything: anchor ANCHOR_ORDER[i] has its x coordinate inside the window iff s >= t_i (x = 360 sigmoid(x_lo +
    g_i (s - t_i)) reaches the window's upper edge only beyond every s), so the frame's count is #{i: s >= t_i}.  The thresholds sit in the widest gaps of the
    batch's scores between consecutive clip maxima, so the clips' track counts (max over frames) take every value 1..5.  y, w and h get
    the default weights with bias 0 (inside their windows).  mode "single": only the first anchor can be valid; "fallback": none."""
    from oracle.ma import _mlp
    ps = (0.3, 0.2, 0, 0)
    keeps = [keep.get("det0"), keep.get("det1"), None, None] if train else None
    h8 = _mlp(P, "detector.detector_net", (0, 3, 6, 8), feats, ("relu",) * 4, keeps, ps).reshape(BB * TT, -1)
    gen = torch.Generator().manual_seed(1007)
    u = torch.randn(h8.shape[1], generator=gen, dtype=torch.float64)
    hm = h8.mean(0)
    u -= (u @ hm) / (hm @ hm) * hm           # s centred on 0: the last layer's products and bias do not cancel (h8 >= 0 has a large mean)
    s = h8 @ u
    srt = s.sort().values
    span = float(srt[-1] - srt[0])
    clip_max = s.view(BB, TT).max(1).values.sort().values

    def gap_mid(a, b):
        inside = srt[(srt > a) & (srt < b)]
        pts = torch.cat([torch.tensor([a, b], dtype=torch.float64), inside]).sort().values
        i = int((pts[1:] - pts[:-1]).argmax())
        return float(pts[i] + pts[i + 1]) / 2

    bounds = [gap_mid(float(clip_max[j - 1]), float(clip_max[j])) for j in (2, 9, 16, 23, 28)]   # clip-max groups -> ntr 1..5
    enabled = {"mixed": 5, "single": 1, "fallback": 0}[mode]
    x_lo = _logit(LO[0] / SCALE[0])                          # the x window is [x_lo, -x_lo] in logits
    W = P["detector.detector_net.10.weight"].clone()
    bias = torch.zeros(20, dtype=torch.float64)
    top = float(srt[-1]) + span
    for i, (a, t) in enumerate(zip(ANCHOR_ORDER, bounds)):
        if i >= enabled:                                     # never valid: x saturates at 0 px
            W[4 * a], bias[4 * a] = 0.0, -30.0
            continue
        g = 2 * abs(x_lo) / (top - t)                        # raw_x = x_lo + g (s - t): x_lo at s = t, -x_lo a span above the top score
        W[4 * a] = g * u
        bias[4 * a] = x_lo - g * t
    return W.float(), bias.float()


def _near_kinks(P, feats):
    """Frames (B,T) / clips (B) with a ReLU pre-activation of the detector / direct classifier (train and eval masks) closer to 0 than
    KINK_MARGIN of its sum of |terms|: there fp32 and fp64 may take different sides of the kink, and the gradient jumps."""
    import torch.nn.functional as F
    bad_f, bad_c = torch.zeros(BB, TT, dtype=torch.bool), torch.zeros(BB, dtype=torch.bool)
    for train in (True, False):
        keep = {k: v.double() for k, v in _keep(train).items()}
        for prefix, x, names, bad in (("detector.detector_net", feats, ("det0", "det1"), bad_f),
                                      ("direct_classifier", feats.mean(1), ("cls0", "cls1"), bad_c)):
            h = x
            for i, li in enumerate((0, 3, 6, 8)):
                W, b = P[f"{prefix}.{li}.weight"], P[f"{prefix}.{li}.bias"]
                pre = F.linear(h, W, b)
                bad |= (pre.abs() < KINK_MARGIN * (F.linear(h.abs(), W.abs()) + b.abs())).any(-1)
                h = F.relu(pre)
                if i < 2 and train:
                    h = h * keep[names[i]] / (1.0 - (0.3, 0.2)[i])
    return bad_f, bad_c


def _tail_case(dev, train, mode):
    """The model, its fp32 state, the features (a leaf), eps / keep-masks, labels: everything both sides consume."""
    from cvad_b200.ma import CausalAnomalyDetector
    torch.manual_seed(4242)
    m = CausalAnomalyDetector()
    P = {k: v.detach().clone() for k, v in m.state_dict().items()}
    P64 = {k: v.double() for k, v in P.items()}
    gen = torch.Generator().manual_seed(1001)
    offset = torch.linspace(-2.0, 2.0, BB).view(BB, 1, 1) * torch.randn(1, 1, FEAT, generator=gen)    # per-clip feature offset
    feats = (torch.randn(BB, TT, FEAT, generator=gen) + offset).float()
    for _ in range(100):                     # redraw the frames (a frame of the clips) that sit on a ReLU kink
        bad_f, bad_c = _near_kinks(P64, feats.double())
        bad_f[bad_c, 0] = True
        if not bad_f.any():
            break
        feats[bad_f] = (torch.randn(int(bad_f.sum()), FEAT, generator=gen) + offset.expand(BB, TT, FEAT)[bad_f]).float()
    assert not bad_f.any()
    eps = torch.randn(BB, MAXDET, NF, generator=gen)
    labels = torch.randint(0, 2, (BB,), generator=gen)
    keep = _keep(train)
    W, b = _engineer_head(P64, feats.double(), {k: v.double() for k, v in keep.items()}, train, mode)
    P["detector.detector_net.10.weight"], P["detector.detector_net.10.bias"] = W, b
    m.load_state_dict(P, strict=True)
    return m, P, feats, eps, keep, labels


class _ProjectionsOnDevice:
    """torch.nn.functional whose linear takes the values of the two 6144-wide projections (K >= 2048) from the project's tensor-core GEMM
    (3xTF32, csrc/gemm_tf32x3_tc.cu) applied to the same inputs; gradients stay plain fp32 on the CPU.  The tensor cores' accumulation is
    not IEEE fp32, so this is "the same fp32 computation" the kernels do there."""

    def __init__(self, dev):
        self.dev = dev

    def __getattr__(self, name):
        return getattr(torch.nn.functional, name)

    def linear(self, x, w, b=None):
        from cvad_b200 import ops
        y = torch.nn.functional.linear(x, w, b)
        if x.dtype != torch.float32 or w.shape[1] < 2048:
            return y
        with torch.no_grad():
            yd = ops.linear_act(x.detach().to(self.dev), w.detach().to(self.dev), None if b is None else b.detach().to(self.dev))
            yd = yd.reshape(y.shape).cpu()
        return y + (yd - y).detach()


def _oracle_tail(dev, P, feats, eps, keep, labels, train, dtype):
    """oracle.ma.ma_tail (+ ma_loss and its backward when training) in ``dtype``.  In fp32 it is the yardstick, so the two 6144-wide
    projections take their values from the tensor-core GEMM."""
    from unittest import mock
    from oracle import ma as o
    with mock.patch.object(o, "F", _ProjectionsOnDevice(dev) if dtype == torch.float32 else o.F):
        return _oracle_tail_run(o, P, feats, eps, keep, labels, train, dtype)


def _oracle_tail_run(o, P, feats, eps, keep, labels, train, dtype):
    names = [k for k in P if not k.startswith("backbone.") and P[k].is_floating_point()]
    Pg = {k: (v.to(dtype).clone().requires_grad_(True) if k in names else v.to(dtype)) for k, v in P.items()}
    f = feats.to(dtype).clone().requires_grad_(train)
    with torch.set_grad_enabled(train):
        out = o.ma_tail(Pg, f, eps.to(dtype), train, {k: v.to(dtype) for k, v in keep.items()})
        if train:
            loss, _ = o.ma_loss(out, labels)
            loss.backward()
    grads = {k: Pg[k].grad for k in names} if train else {}
    return out, f.grad, grads


def _coverage(cnt, ntr):
    """The edges the engineered batch must contain."""
    cnt, ntr = cnt.long(), ntr.long()
    assert set(ntr.tolist()) == {1, 2, 3, 4, 5}, ntr.tolist()
    c = cnt.view(BB, TT)                                                      # counts before the clamp to 1
    assert ((c == 0).any(1) & (c > 0).any(1)).any()                           # a clip with fallback frames beside real detections
    assert (cnt.view(BB, TT).min(1).values < ntr).any()                       # a track present in some frames, zero-padded in others


def _margin_px(P, feats, keep, train):
    """Distance of every box coordinate from its window's edges, in fp64."""
    from oracle.ma import _mlp
    keeps = [keep["det0"].double(), keep["det1"].double(), None, None, None] if train else None
    Pd = {k: v.double() for k, v in P.items()}
    raw = _mlp(Pd, "detector.detector_net", (0, 3, 6, 8, 10), feats.double(), ("relu", "relu", "relu", "relu", None), keeps,
               (0.3, 0.2, 0, 0, 0)).view(BB, TT, MAXDET, 4)
    box = torch.sigmoid(raw) * torch.tensor(SCALE, dtype=torch.float64) + torch.tensor(OFF, dtype=torch.float64)
    lo, hi = torch.tensor(LO, dtype=torch.float64), torch.tensor(HI, dtype=torch.float64)
    valid = ((box >= lo) & (box <= hi)).all(-1)
    return float(torch.minimum((box - lo).abs(), (box - hi).abs()).min()), valid.sum(-1)


@pytest.mark.parametrize("train,mode", [(True, "mixed"), (False, "mixed"), (True, "fallback"), (True, "single")])
def test_tail_vs_fp64_oracle(dev, train, mode):
    """The whole branch behind the backbone through model.tail() vs oracle.ma.ma_tail in fp64: counts exact, values and every tail
    gradient (and the features' gradient) elementwise within the yardstick bound; groups whose reference gradient is None get none."""
    from cvad_b200.ma import SLOT_DETECTOR, SLOT_STRUCTURE, MATrainer
    from cvad_b200.noise import FixedNoise
    m, P, feats, eps, keep, labels = _tail_case(dev, train, mode)
    margin, raw_cnt = _margin_px(P, feats, keep, train)
    assert margin >= MARGIN_PX, margin
    if mode == "mixed":
        _coverage(raw_cnt, raw_cnt.clamp(min=1).max(1).values)
    elif mode == "fallback":
        assert (raw_cnt == 0).all()
    else:
        assert (raw_cnt <= 1).all() and (raw_cnt == 1).any()
    tr = MATrainer(m, dev, precision="fp32")
    tr.model.train(train)
    tr.model.noise = FixedNoise({"eps": eps.to(dev), **{k: v.to(dev) for k, v in keep.items()}})
    tr.optimizer.zero_grad()
    f = feats.to(dev).requires_grad_(train)
    with torch.set_grad_enabled(train):
        out = tr.model.tail(f)
        if train:
            loss, _ = tr.loss_on_device(out, labels.to(dev))
            loss.backward()
    torch.cuda.synchronize()
    r64, fg64, g64 = _oracle_tail(dev, P, feats, eps, keep, labels, train, torch.float64)
    r32, fg32, g32 = _oracle_tail(dev, P, feats, eps, keep, labels, train, torch.float32)
    d = out["dense"]
    assert torch.equal(d["det_counts"].cpu().long(), r64["det_counts"]) and torch.equal(r32["det_counts"], r64["det_counts"])
    assert torch.equal(d["n_tracks"].cpu().long(), r64["n_tracks"])
    if mode == "mixed":
        _coverage(raw_cnt, d["n_tracks"].cpu())
    tag = f"{'train' if train else 'eval'}/{mode}"
    act = torch.arange(MAXDET).view(1, -1) < r64["n_tracks"].view(-1, 1)
    check_yard(f"tail {tag} detections", d["detections"], r64["detections"], r32["detections"])
    check_yard(f"tail {tag} z (active tracks)", d["causal_factors"].cpu()[act], r64["causal_factors"][act], r32["causal_factors"][act])
    assert (d["causal_factors"].cpu()[~act] == 0).all()
    check_yard(f"tail {tag} kl", d["kl_losses"], r64["kl_losses"], r32["kl_losses"])
    check_yard(f"tail {tag} adjacency", d["adjacency_matrices"], r64["adjacency_matrices"], r32["adjacency_matrices"])
    for k in ("causal_anomaly_scores", "direct_predictions", "anomaly_scores"):
        check_yard(f"tail {tag} {k}", out[k].detach(), r64[k].detach(), r32[k].detach())
    if not train:
        return
    check_yard(f"tail {tag} features.grad", f.grad, fg64, fg32)
    params = dict(tr.model.named_parameters())
    for k, g in g64.items():
        got = params[k].grad
        none = g is None or (float(g.abs().max()) == 0.0 and ("detector" in k or "structure_learner" in k))   # oracle/train.py's rule
        if none:
            assert got is None or (got == 0).all(), k
            continue
        check_yard(f"tail {tag} grad {k}", got, g, g32[k])
    flags = tr.optimizer.arena.header.cpu()
    det_none = all(g64[k] is None or float(g64[k].abs().max()) == 0 for k in g64 if k.startswith("detector."))
    str_none = all(g64[k] is None or float(g64[k].abs().max()) == 0 for k in g64
                   if k.startswith("structure_learner.node_encoder") or k.startswith("structure_learner.edge_predictor"))
    assert det_none == (mode == "fallback") and str_none == (mode != "mixed")
    assert float(flags[SLOT_DETECTOR]) == (0.0 if det_none else 1.0)
    assert float(flags[SLOT_STRUCTURE]) == (0.0 if str_none else 1.0)
