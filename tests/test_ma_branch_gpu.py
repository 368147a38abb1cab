"""M-A's causal branch behind the GRU as one fused op (csrc/ma_branch.cu through ma_ops.causal_branch) against float64.

The reference is oracle.ma.ma_tail itself, run from the GRU's last state: its gru_last returns the test's hT, its detect returns counts that
give every clip the chosen track count, and its 6144-wide linears (the direct classifier, not part of the branch) return zeros.  Everything
the fused op computes -- encoder Linear, factor MLP, heads, reparameterisation, KL, node encoder, edge MLP, adjacency, structured,
dynamics, scorer inputs, the three scorers with the scorer0 keep-mask and their combination -- runs through the oracle's own code.

Bounds are the yardstick of test_ma_tail_gpu.py: the kernel's error <= 4 x the error of the same computation in fp32 on the CPU plus 64
fp32 ulps of the tensor's scale, both against float64.  Clips in which a ReLU input or cur - prd (the |.| of the scorer inputs) lies within
KINK_MARGIN of 0, relative to its sum of |terms|, are redrawn: there fp32 and fp64 may take different sides of the kink.
"""
import math
from unittest import mock

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

MAXDET, NF, HID = 5, 6, 64
KINK_MARGIN = 1e-5
STRUCTURE = ("structure_learner.node_encoder.", "structure_learner.edge_predictor.")


def ulp32(scale):
    return float(np.spacing(np.float32(max(scale, 1e-30))))


def check_yard(name, got, ref, cpu32):
    got, ref, cpu32 = (torch.as_tensor(v).double().cpu() for v in (got, ref, cpu32))
    assert torch.isfinite(got).all(), f"{name}: non-finite output"
    err = float((got - ref).abs().max()) if got.numel() else 0.0
    yard = float((cpu32 - ref).abs().max()) if got.numel() else 0.0
    scale = float(ref.abs().max()) if got.numel() else 0.0
    bound = 4.0 * yard + 64.0 * ulp32(scale)
    ratio = err / bound if bound > 0 else (0.0 if err == 0 else math.inf)
    print(f"[ma_branch] {name}: err {err:.3e} yardstick {yard:.3e} scale {scale:.3e} err/bound {ratio:.3f}")
    assert ratio <= 1.0, (name, err, yard, scale)


class _OracleF:
    """torch.nn.functional for the oracle run: the 6144-wide linears return zeros, and while ``on`` every clip with a ReLU input (or a
    cur - prd entering the causal scorer) within KINK_MARGIN of 0 relative to its sum of |terms| is marked in ``bad``."""

    def __init__(self, B):
        self.bad = torch.zeros(B, dtype=torch.bool)
        self.on = False
        self.last = None

    def __getattr__(self, name):
        return getattr(F, name)

    def linear(self, x, w, b=None):
        if w.shape[1] >= 2048:
            return torch.zeros(*x.shape[:-1], w.shape[0], dtype=x.dtype)
        y = F.linear(x, w, b)
        if self.on:
            xd = x.detach()
            self.last = (y, F.linear(xd.abs(), w.detach().abs(), None if b is None else b.detach().abs()))
            if w.shape[1] == 3 * NF:                     # the causal scorer's input [cur | prd | |cur - prd|]
                cur, prd = xd[..., :NF], xd[..., NF:2 * NF]
                self.bad |= ((cur - prd).abs() < KINK_MARGIN * (cur.abs() + prd.abs())).reshape(x.shape[0], -1).any(1)
        return y

    def relu(self, h):
        if self.on and self.last is not None and h is self.last[0]:
            self.bad |= (h.detach().abs() < KINK_MARGIN * self.last[1]).reshape(h.shape[0], -1).any(1)
        return F.relu(h)


def oracle_branch(P, names, hT, ntr, eps, keep, train, dtype, ups=None):
    """(z, kl, adj, causal), the gradients of sum(out * up) w.r.t. hT and the branch parameters ``names``, and the clips near a kink."""
    from oracle import ma as o
    B = ntr.shape[0]
    Pd = {k: (v.to(dtype).clone().requires_grad_(ups is not None) if k in names else v.to(dtype)) for k, v in P.items()}
    h = hT.to(dtype).clone().requires_grad_(ups is not None)
    fo = _OracleF(B)

    def gru_last(_P, _x):
        fo.on = True
        return h

    def detect(_P, feats, _train, _keep):
        return torch.zeros(B, 1, MAXDET, 4, dtype=dtype), ntr.long().view(B, 1)

    with mock.patch.object(o, "F", fo), mock.patch.object(o, "gru_last", gru_last), mock.patch.object(o, "detect", detect), \
            torch.set_grad_enabled(ups is not None):
        out = o.ma_tail(Pd, torch.zeros(B, 1, 1, dtype=dtype), eps.to(dtype), train, {"scorer0": keep.to(dtype)} if train else {})
        res = (out["causal_factors"], out["kl_losses"], out["adjacency_matrices"], out["causal_anomaly_scores"])
        if ups is None:
            return tuple(r.detach() for r in res), None, fo.bad
        act = (torch.arange(MAXDET).view(1, -1, 1) < ntr.long().view(-1, 1, 1)).to(dtype)
        loss = sum((r * (u.to(dtype) * (act if i == 0 else 1))).sum() for i, (r, u) in enumerate(zip(res, ups)) if u is not None)
        loss.backward()
    return tuple(r.detach() for r in res), {"hT": h.grad, **{k: Pd[k].grad for k in names}}, fo.bad


def make_case(B, train, seed, ntr=None):
    from cvad_b200.ma import CausalAnomalyDetector
    torch.manual_seed(seed)
    m = CausalAnomalyDetector()
    gen = torch.Generator().manual_seed(seed)
    if ntr is None:
        ntr = torch.randint(1, MAXDET + 1, (B,), generator=gen, dtype=torch.int32)
        ntr[: min(B, MAXDET)] = torch.arange(1, min(B, MAXDET) + 1, dtype=torch.int32)
    hT = torch.rand(B * MAXDET, HID, generator=gen) * 2 - 1
    eps = torch.randn(B, MAXDET, NF, generator=gen)
    keep = (torch.rand(B, 64, generator=gen) >= 0.2).float()
    P = {k: v.detach().clone() for k, v in m.state_dict().items()}
    ids = {id(p): n for n, p in m.named_parameters()}
    names = [ids[id(p)] for p in m.causal_branch_params()]
    for _ in range(50):                      # redraw the states of clips that sit on a kink
        _, _, bad = oracle_branch(P, names, hT, ntr, eps, keep, train, torch.float64)
        if not bad.any():
            break
        idx = bad.nonzero().flatten()
        hT.view(B, MAXDET, HID)[idx] = torch.rand(len(idx), MAXDET, HID, generator=gen) * 2 - 1
    assert not bad.any()
    return m, P, names, hT, ntr, eps, keep, gen


def _device_params(m, dev):
    m = m.to(dev)
    return m, m.causal_branch_params()


@pytest.mark.parametrize("B", [1, 32, 300, 5000])
@pytest.mark.parametrize("train", [True, False])
@pytest.mark.parametrize("upstream", ["all", "loss"])
def test_branch_vs_fp64_oracle(dev, B, train, upstream):
    """Values and every gradient elementwise against the fp64 oracle; every track count 1..5 in one batch; inactive z slots and dhT rows
    exactly 0; parameter gradients are ADDED to a pre-filled .grad.  upstream "all": random gradients on z, kl, adj and the causal score;
    "loss": only on kl and the causal score, as the training loss sends them."""
    from cvad_b200 import ma_ops
    m, P, names, hT, ntr, eps, keep, gen = make_case(B, train, 4100 + B + 7 * train)
    ups = [torch.randn(B, MAXDET, NF, generator=gen), torch.randn(B, generator=gen), torch.randn(B, NF, NF, generator=gen),
           torch.randn(B, generator=gen)]
    if upstream == "loss":
        ups[0] = ups[2] = None
    r64, g64, _ = oracle_branch(P, names, hT, ntr, eps, keep, train, torch.float64, ups)
    r32, g32, _ = oracle_branch(P, names, hT, ntr, eps, keep, train, torch.float32, ups)
    m, params = _device_params(m, dev)
    pre = {n: torch.randn(p.shape, generator=gen) * 0.01 for n, p in zip(names, params)}
    for n, p in zip(names, params):
        p.grad = pre[n].to(dev)
    h = hT.to(dev).requires_grad_(True)
    out = ma_ops.causal_branch(h, ntr.to(dev), eps.to(dev), keep.to(dev) if train else None, params)
    act = torch.arange(MAXDET).view(1, -1) < ntr.long().view(-1, 1)
    tag = f"B{B} {'train' if train else 'eval'} {upstream}"
    z = out[0].detach().cpu()
    assert (z[~act] == 0).all()
    check_yard(f"{tag} z", z[act], r64[0][act], r32[0][act])
    for i, name in ((1, "kl"), (2, "adj"), (3, "causal")):
        check_yard(f"{tag} {name}", out[i].detach(), r64[i], r32[i])
    adj = out[2].detach().cpu()
    live = act.unsqueeze(2) & act.unsqueeze(1)
    live[:, torch.arange(MAXDET), torch.arange(MAXDET)] = False
    assert (adj[:, :MAXDET, :MAXDET][~live] == 0).all() and (adj[:, MAXDET] == 0).all() and (adj[:, :, MAXDET] == 0).all()
    torch.autograd.backward([o for o, u in zip(out, ups) if u is not None], [u.to(dev) for u in ups if u is not None])
    torch.cuda.synchronize()
    dh = h.grad.cpu().view(B, MAXDET, HID)
    assert (dh[~act] == 0).all()
    check_yard(f"{tag} dhT", dh, g64["hT"].view(B, MAXDET, HID), g32["hT"].view(B, MAXDET, HID))
    for n, p in zip(names, params):
        check_yard(f"{tag} grad {n}", p.grad, pre[n].double() + g64[n], pre[n] + g32[n])


def test_branch_abi_writes_every_output(dev):
    """The entry points on NaN-filled outputs: every slot of z, kl, adj, causal and dhT is written and equals the autograd op's result;
    NULL upstream gradients are zeros; a NULL gradient pointer leaves that buffer untouched."""
    from cvad_b200 import ma_ops
    from cvad_b200.ops import _ptr_array
    B = 37
    m, P, names, hT, ntr, eps, keep, gen = make_case(B, True, 4300)
    m, params = _device_params(m, dev)
    hd, nd, ed, kd = hT.to(dev), ntr.to(dev), eps.to(dev), keep.to(dev)
    z, kl, adj, causal = (torch.full(s, float("nan"), device=dev) for s in ((B, MAXDET, NF), (B,), (B, NF, NF), (B,)))
    call = lambda name, *a: ma_ops._call(name, *[x.data_ptr() if isinstance(x, torch.Tensor) else x for x in a])
    pa = _ptr_array(params)
    call("cvad_ma_branch_fwd_f32", hd, nd, ed, kd, B, pa, z, kl, adj, causal, torch.cuda.current_stream().cuda_stream)
    with torch.no_grad():
        ref = ma_ops.causal_branch(hd, nd, ed, kd, params)
    for got, want in zip((z, kl, adj, causal), ref):
        assert torch.equal(got, want)
    dkl, dc = torch.randn(B, generator=gen).to(dev), torch.randn(B, generator=gen).to(dev)
    grads = [torch.zeros_like(p) for p in params]
    grads[3] = torch.full_like(params[3], 7.0)          # this parameter "needs no gradient": NULL pointer, buffer untouched
    ptrs = [g for g in grads]
    ptrs[3] = None
    dhT = torch.full((B * MAXDET, HID), float("nan"), device=dev)
    call("cvad_ma_branch_bwd_f32", hd, nd, ed, kd, B, pa, None, dkl, None, dc, dhT, _ptr_array(ptrs), torch.cuda.current_stream().cuda_stream)
    h = hd.clone().requires_grad_(True)
    for p in params:
        p.grad = None
    out = ma_ops.causal_branch(h, nd, ed, kd, params)
    torch.autograd.backward([out[1], out[3]], [dkl, dc])
    assert torch.equal(dhT, h.grad)
    assert (grads[3] == 7.0).all()
    for i, (g, p) in enumerate(zip(grads, params)):
        if i != 3:
            assert torch.allclose(g, p.grad, rtol=1e-5, atol=1e-6 * float(p.grad.abs().max()) + 1e-30), names[i]
    dh0 = torch.full_like(dhT, float("nan"))
    g0 = [torch.zeros_like(p) for p in params]
    call("cvad_ma_branch_bwd_f32", hd, nd, ed, kd, B, pa, None, None, None, None, dh0, _ptr_array(g0), torch.cuda.current_stream().cuda_stream)
    assert (dh0 == 0).all() and all((g == 0).all() for g in g0)


def test_structure_gradients_exactly_zero_single_track(dev):
    """Every clip with one track: no live edge pair, so the node encoder and the edge MLP receive exact zeros (their group's activity flag
    stays with traj_assemble); every other gradient matches the oracle."""
    from cvad_b200 import ma_ops
    B = 300
    m, P, names, hT, ntr, eps, keep, gen = make_case(B, True, 4400, ntr=torch.ones(B, dtype=torch.int32))
    ups = [torch.randn(B, MAXDET, NF, generator=gen), torch.randn(B, generator=gen), torch.randn(B, NF, NF, generator=gen),
           torch.randn(B, generator=gen)]
    r64, g64, _ = oracle_branch(P, names, hT, ntr, eps, keep, True, torch.float64, ups)
    r32, g32, _ = oracle_branch(P, names, hT, ntr, eps, keep, True, torch.float32, ups)
    m, params = _device_params(m, dev)
    h = hT.to(dev).requires_grad_(True)
    out = ma_ops.causal_branch(h, ntr.to(dev), eps.to(dev), keep.to(dev), params)
    assert (out[2] == 0).all()
    torch.autograd.backward(list(out), [u.to(dev) for u in ups])
    for n, p in zip(names, params):
        if n.startswith(STRUCTURE):
            assert (p.grad == 0).all(), n
        else:
            check_yard(f"single-track grad {n}", p.grad, g64[n], g32[n])


def test_graph_replay_matches_eager(dev):
    """Forward + backward captured in one CUDA graph: the replay's outputs and dhT equal eager bit for bit; the parameter gradients
    (summed across CTAs in an unspecified order) agree to a few ulps."""
    from cvad_b200 import ma_ops
    B = 32
    m, P, names, hT, ntr, eps, keep, gen = make_case(B, True, 4500)
    m, params = _device_params(m, dev)
    hd, nd, ed, kd = hT.to(dev), ntr.to(dev), eps.to(dev), keep.to(dev)
    ups = [torch.randn(B, generator=gen).to(dev), torch.randn(B, generator=gen).to(dev)]

    def step():
        for p in params:
            p.grad.zero_()
        h = hd.detach().requires_grad_(True)
        out = ma_ops.causal_branch(h, nd, ed, kd, params)
        torch.autograd.backward([out[1], out[3]], ups)
        return [o.detach() for o in out] + [h.grad]

    for p in params:
        p.grad = torch.zeros_like(p)
    eager = [t.clone() for t in step()]
    eager_g = [p.grad.clone() for p in params]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        static = step()
    g.replay()
    torch.cuda.synchronize()
    for a, b in zip(static, eager):
        assert torch.equal(a, b)
    for n, p, e in zip(names, params, eager_g):
        assert float((p.grad - e).abs().max()) <= 64 * ulp32(float(e.abs().max())), n
