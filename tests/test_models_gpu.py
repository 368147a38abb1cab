"""Model-level parity on the B200 against the golden fixtures produced by the reference (tests/golden) and the oracle."""
import copy
import os

import numpy as np
import pytest
import torch

import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rel(a, b, floor=1e-3):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).abs().max() / max(float(b.abs().max()), floor))


# --------------------------------------------------------------------------------------------------------- M-B
def test_mb_eval_parity_fp32(dev, gold):
    """a1-a3: scores / adjacency / features within 1e-5 relative (north-star fp32 tolerance), identical ranking."""
    from cvad_b200.mb import CausalAnomalyDetector
    g = gold("mb.pt")
    m = CausalAnomalyDetector().to(dev)
    m.load_state_dict(gold("best_improved_model.pth")["model_state_dict"], strict=True)
    m.eval()
    for c in g["eval"]:
        x = (synth.mb_clips_bright if c["bright"] else synth.mb_clips)(c["B"], c["T"], c["H"], c["W"], c["seed"])
        with torch.no_grad():
            s, a, f = m(x.to(dev))
        assert s.shape == (c["B"], 1) and a.shape == (c["B"], 16, 16) and f.shape == (c["B"], 16)
        assert rel(s, c["scores"]) < 1e-5, (c, rel(s, c["scores"]))
        assert rel(a, c["adj"]) < 1e-5
        assert rel(f, c["feat"]) < 1e-5
        assert torch.equal(((a.cpu() > 0.1).sum((1, 2))), (c["adj"] > 0.1).sum((1, 2)))
    ka = g["known_answers"]["scores_T8"]
    x = synth.mb_clips(4, 8, 64, 64, 1234)
    with torch.no_grad():
        s, _, _ = m(x.to(dev))
    assert rel(s.flatten(), torch.tensor(ka)) < 1e-5


def test_mb_train_step_parity(dev, gold):
    """a4-a5: loss, the 7 components and every parameter gradient of one training forward/backward."""
    from cvad_b200.mb import COMPONENT_KEYS, ImprovedMiniCausalVAD
    from cvad_b200.noise import FixedNoise
    g = gold("mb.pt")
    ck = gold("best_improved_model.pth")
    for c in g["train"]:
        tr = ImprovedMiniCausalVAD(device=dev, verbose=False)
        tr.model.load_state_dict(ck["model_state_dict"], strict=True)
        tr.model.train()
        tr.model.noise = FixedNoise({"feat": c["keep_feat"], "graph": c["keep_graph"]})
        x = synth.mb_clips_bright(c["B"], c["T"], 64, 64, c["seed"]).to(dev)
        tr.optimizer.zero_grad()
        s, a, f = tr.model(x)
        loss, comp = tr.loss_on_device(s, a, torch.zeros(c["B"], device=dev), c["pseudo"].to(dev))
        loss.backward()
        assert rel(loss, c["loss"]) < 1e-5
        for i, k in enumerate(COMPONENT_KEYS):
            assert abs(float(comp[i + 1]) - c["comps"][k]) <= 1e-5 * max(1.0, abs(c["comps"][k])), k
        assert rel(s, c["scores"]) < 1e-5 and rel(a, c["adj"]) < 1e-5
        for k, p in tr.model.named_parameters():
            sm = c["grad_summary"][k]
            assert abs(float(p.grad.double().norm()) - sm["norm"]) <= 2e-4 * max(sm["norm"], 1e-7), k
            assert rel(p.grad.flatten()[:16], sm["head"], floor=sm["absmax"] + 1e-12) < 2e-4, k
            if c["grads"][k] is not None:
                assert rel(p.grad, c["grads"][k], floor=sm["absmax"] + 1e-12) < 2e-4, k


def test_mb_trajectory_from_shipped_checkpoint(dev, gold, tmp_path):
    """3 optimizer steps from best_improved_model.pth incl. its AdamW state == the reference's trajectory (s2:221-238)."""
    from cvad_b200.mb import ImprovedMiniCausalVAD
    from cvad_b200.noise import FixedNoise
    g = gold("mb.pt")["trajectory"]
    ck = gold("best_improved_model.pth")
    tr = ImprovedMiniCausalVAD(device=dev, verbose=False)
    tr.model.load_state_dict(ck["model_state_dict"], strict=True)
    tr.optimizer.load_state_dict(copy.deepcopy(ck["optimizer_state_dict"]))
    tr.model.train()
    for it, sd in enumerate(g["seeds"]):
        x = synth.mb_clips_bright(8, 8, 64, 64, sd).to(dev)
        tr.model.noise = FixedNoise({"feat": synth.keep_mask((8, 16), 0.3, sd + 1), "graph": synth.keep_mask((8, 128), 0.3, sd + 2)})
        pseudo = (g["steps"][it]["u"] > 0.95).float().to(dev)
        comp = tr.train_step(x, torch.zeros(8, device=dev), pseudo)
        assert abs(float(comp[0]) - g["losses"][it]) < 2e-5 * max(1, abs(g["losses"][it])), it
        assert abs(tr.optimizer.last_grad_norm() - g["steps"][it]["grad_norm"]) < 2e-4 * g["steps"][it]["grad_norm"]
    sd = tr.model.state_dict()
    for k, v in g["final_small"].items():
        assert rel(sd[k], v) < 2e-5, k
    for k, sm in g["final_summary"].items():
        assert abs(float(sd[k].double().norm()) - sm["norm"]) < 1e-5 * max(sm["norm"], 1e-6), k
    osd = tr.optimizer.state_dict()
    assert float(osd["state"][0]["step"]) == g["final_opt_step"]
    # checkpoint round trip through stock torch (s2:437-443 layout)
    path = tmp_path / "cvad_roundtrip.pth"
    torch.save({"model_state_dict": tr.model.state_dict(), "optimizer_state_dict": osd, "epoch": 0, "eval_metrics": {}}, path)
    back = torch.load(path, map_location="cpu", weights_only=False)
    ref_opt_keys = set(ck["optimizer_state_dict"]["param_groups"][0].keys())
    assert set(back["optimizer_state_dict"]["param_groups"][0].keys()) == ref_opt_keys
    stock = torch.optim.AdamW([torch.nn.Parameter(v.clone()) for v in back["model_state_dict"].values()], lr=5e-4, weight_decay=1e-3)
    stock.load_state_dict(back["optimizer_state_dict"])


def test_mb_epoch_api_and_nan_skip(dev, gold, tmp_path):
    from cvad_b200.mb import ImprovedMiniCausalVAD, MiniCausalVAD
    tr = ImprovedMiniCausalVAD(device=dev, verbose=False)
    tr.model.load_state_dict(gold("best_improved_model.pth")["model_state_dict"], strict=True)
    loader = [(synth.mb_clips_bright(4, 8, 64, 64, 200 + i), torch.zeros(4)) for i in range(3)]
    avg, comps = tr.train_epoch_improved(loader)
    assert set(comps) == {"anomaly_loss", "acyclicity_loss", "sparsity_loss", "consistency_loss", "structure_loss", "edge_count",
                          "sparsity_ratio"}
    assert avg == avg and avg > 0
    preds, graphs, metrics = tr.evaluate_improved(loader)
    assert preds.shape == (12,) and graphs.shape == (12, 16, 16) and len(metrics) == 8
    before = {k: v.clone() for k, v in tr.model.state_dict().items()}
    bad = loader[0][0].clone()
    bad[0, 0, 0, 0, 0] = float("nan")
    tr.model.train()
    tr.train_step(bad.to(dev), torch.zeros(4, device=dev))
    assert tr.optimizer.skipped_steps() == 1
    for k, v in tr.model.state_dict().items():
        assert torch.equal(v, before[k]), k
    m = MiniCausalVAD(device=dev)
    loss, c4 = m.train_epoch(loader)
    assert set(c4) == {"anomaly_loss", "acyclicity_loss", "sparsity_loss", "consistency_loss"}
    p, _, gr = m.evaluate(loader)
    assert p.shape == (12,) and gr.shape == (12, 16, 16)
    m.save_model(tmp_path / "cvad_mini.pth")
    m.load_model(tmp_path / "cvad_mini.pth")
    for pg in m.optimizer.param_groups:
        pg["lr"] = 1e-4          # s1:104-106


# --------------------------------------------------------------------------------------------------------- M-C
def _mc_synth(g):
    st = synth.synth_fill(g["init_state"], seed=g["state_seed"])
    for k in st:
        if k.startswith("classifier") and k.endswith("weight"):
            st[k] = st[k] * 3.0
    return st


def test_mc_eval_parity(dev, gold):
    from cvad_b200.mc import SimpleVideoAnomalyDetector
    g = gold("mc.pt")
    m = SimpleVideoAnomalyDetector().to(dev)
    for c in g["eval"]:
        m.load_state_dict(g["init_state"] if c["weights"] == "init" else _mc_synth(g), strict=True)
        m.eval()
        x = synth.mc_clips(c["B"], c["T"], c["H"], c["W"], c["seed"]).to(dev)
        with torch.no_grad():
            s = m(x)
        assert s.shape == (c["B"], 1)
        assert rel(s, c["scores"]) < 1e-5, c


def test_mc_train_step_parity(dev, gold):
    from cvad_b200 import ops
    from cvad_b200.mc import SimpleVideoAnomalyDetector
    from cvad_b200.noise import FixedNoise
    g = gold("mc.pt")
    for c in g["train"]:
        m = SimpleVideoAnomalyDetector().to(dev)
        m.load_state_dict(_mc_synth(g), strict=True)
        m.train()
        m.noise = FixedNoise({"cls0": c["keep0"], "cls1": c["keep1"]})
        x = synth.mc_clips(c["B"], c["T"], 64, 64, c["seed"]).to(dev)
        s = m(x)
        loss = ops.bce_loss(s.reshape(-1), c["y"].to(dev))
        loss.backward()
        assert rel(loss, c["loss"]) < 1e-5
        assert rel(s, c["scores"]) < 1e-5
        gscale = max(float(v.abs().max()) for v in c["grads"].values())
        for k, p in m.named_parameters():
            assert rel(p.grad, c["grads"][k], floor=gscale) < 2e-4, k
        sd = m.state_dict()
        for k, v in c["new_stats"].items():
            assert rel(sd[k].float(), v.float()) < 1e-5, k


def test_mc_trajectory_and_trainer(dev, gold):
    from cvad_b200.mc import SimpleVideoAnomalyDetector, StableTrainer, roc_auc
    from cvad_b200.noise import FixedNoise
    g = gold("mc.pt")
    tj = g["trajectory"]
    m = SimpleVideoAnomalyDetector()
    m.load_state_dict(_mc_synth(g), strict=True)
    tr = StableTrainer(m, [], [], dev, lr=1e-3)
    tr.model.train()
    for it, sd in enumerate(tj["seeds"]):
        x = synth.mc_clips(4, 8, 64, 64, sd).to(dev)
        y = (torch.rand(4, generator=synth.gen(sd + 5)) > 0.5).float().to(dev)
        tr.model.noise = FixedNoise({"cls0": synth.keep_mask((4, 32), 0.5, sd + 1), "cls1": synth.keep_mask((4, 16), 0.3, sd + 2)})
        loss, _ = tr.train_step(x, y)
        assert abs(float(loss) - tj["losses"][it]) < 1e-4 * max(1, abs(tj["losses"][it])), it
    sd = tr.model.state_dict()
    for k, v in tj["final"].items():
        if k in ("features.0.bias", "features.4.bias", "features.8.bias", "features.1.running_mean", "features.5.running_mean",
                 "features.9.running_mean"):
            # conv biases feeding BatchNorm have an analytically zero gradient: Adam normalises pure round-off noise into
            # +-lr steps, so these (and the BN running means that absorb them) follow a noise-driven walk in the reference
            # too; bound it by the 3 steps taken.
            assert float((sd[k].cpu() - v).abs().max()) <= 2 * 3 * 1e-3 + 1e-6, k
            continue
        # Adam divides by sqrt(v): elements whose gradient is at round-off level move by up to lr per step in either
        # implementation, so 3 steps are compared at 2e-3 of the tensor's largest weight (observed 2e-4), not at 1e-4
        assert rel(sd[k].float(), v.float()) < 2e-3, k
    import numpy as np
    t = np.array([0, 1, 1, 0, 1, 0]); s = np.array([0.1, 0.8, 0.4, 0.4, 0.9, 0.2])
    assert abs(roc_auc(t, s) - (8.5 / 9)) < 1e-12
    loader = [(synth.mc_clips(4, 8, 64, 64, 300 + i), (torch.arange(4) % 2).float()) for i in range(2)]
    tr2 = StableTrainer(SimpleVideoAnomalyDetector(), loader, loader, dev)
    l, a = tr2.train_epoch()
    tl, auc, acc = tr2.evaluate()
    assert l > 0 and 0 <= a <= 1 and 0 <= auc <= 1


# --------------------------------------------------------------------------------------------------------- M-A
def _ma_model(dev, c):
    from test_oracle_golden import ma_noise, ma_synth_state
    from cvad_b200.ma import CausalAnomalyDetector
    from cvad_b200.noise import FixedNoise
    m = CausalAnomalyDetector()
    m.load_state_dict(ma_synth_state(c["seed"], c["live"]), strict=True)
    eps, keep = ma_noise(c)
    noise = FixedNoise({"eps": eps, **keep})
    return m, noise


@pytest.mark.parametrize("idx", [0, 2])
def test_ma_eval_parity_fp32(dev, gold, idx):
    """a7-a15 forward in eval mode (fp32 path): scores, probabilities, KL, adjacency, detections vs the reference."""
    c = gold("ma.pt")["cases"][idx]
    assert not c["train"]
    m, noise = _ma_model(dev, c)
    m = m.to(dev).eval()
    m.noise = noise
    x = synth.ma_clips(c["B"], c["T"], c["H"], c["W"], c["xseed"], c["wide"]).to(dev)
    with torch.no_grad():
        out = m(x)
    assert set(out) >= {"anomaly_scores", "causal_factors", "adjacency_matrices", "kl_losses", "detections", "direct_predictions",
                        "causal_anomaly_scores"}
    assert rel(out["anomaly_scores"], c["anomaly_scores"]) < 2e-5
    assert rel(out["causal_anomaly_scores"], c["causal_anomaly_scores"]) < 2e-5
    assert rel(out["direct_predictions"], c["direct_predictions"]) < 2e-5
    d = out["dense"]
    assert rel(d["kl_losses"], c["kl_losses"]) < 2e-5
    assert rel(d["adjacency_matrices"], c["adjacency"]) < 2e-5
    assert torch.equal(d["det_counts"].cpu().long(), c["det_counts"])
    assert torch.equal(d["n_tracks"].cpu().long(), c["n_tracks"])
    assert rel(d["detections"], c["detections"]) < 2e-5
    assert abs(float(d["features"].double().norm()) - c["features_summary"]["norm"]) < 1e-5 * c["features_summary"]["norm"]
    # ragged views of the reference's output dict
    n = c["n_tracks"].tolist()
    assert len(out["causal_factors"]) == c["B"] and out["causal_factors"][0].shape == (n[0], 6)
    assert len(out["detections"][0]) == c["T"] and out["detections"][0][0].shape == (int(c["det_counts"][0, 0]), 4)
    assert len(out["kl_losses"]) == c["B"] and out["adjacency_matrices"][0].shape == (6, 6)


@pytest.mark.parametrize("idx", [1, 3])
def test_ma_train_step_parity_fp32(dev, gold, idx):
    """a16: 4-term loss, gradients of every parameter, BN running statistics, and the grad-is-None groups."""
    from cvad_b200.ma import MATrainer
    c = gold("ma.pt")["cases"][idx]
    assert c["train"]
    m, noise = _ma_model(dev, c)
    tr = MATrainer(m, dev, precision="fp32")
    tr.model.train()
    tr.model.noise = noise
    x = synth.ma_clips(c["B"], c["T"], c["H"], c["W"], c["xseed"], c["wide"]).to(dev)
    labels = c["labels"].to(dev)
    tr.optimizer.zero_grad()
    out = tr.model(x)
    loss, comp = tr.loss_on_device(out, labels)
    loss.backward()
    assert rel(loss, c["loss"]) < 5e-5
    for i, k in enumerate(("classification", "anomaly", "causal", "kl")):
        assert abs(float(comp[i + 1]) - c["comps"][k]) < 5e-5 * max(1.0, abs(c["comps"][k])), k
    assert rel(out["anomaly_scores"], c["anomaly_scores"]) < 5e-5
    gnorm = max(v["norm"] for v in c["grad_summary"].values())
    for k, p in tr.model.named_parameters():
        if k not in c["grad_summary"]:
            continue
        sm = c["grad_summary"][k]
        if sm["norm"] < 1e-5 * gnorm:
            continue
        got = float(p.grad.double().norm())
        assert abs(got - sm["norm"]) <= 5e-3 * sm["norm"], (k, got, sm["norm"])
        if "full" in sm:
            assert float((p.grad.cpu() - sm["full"]).double().norm()) <= 5e-3 * sm["norm"], k
    sd = tr.model.state_dict()
    for k, v in c["new_stats"].items():
        assert rel(sd[k].float(), v.float()) < 2e-5, k
    # groups whose gradient is None in the reference must not be stepped (no weight decay either)
    before = {k: p.detach().clone() for k, p in tr.model.named_parameters()}
    tr.optimizer.step()
    for k, p in tr.model.named_parameters():
        if not p.requires_grad:
            continue
        moved = not torch.equal(before[k], p.detach())
        if not c["has_grad"][k]:
            assert not moved, k
        elif c["grad_summary"].get(k, {"norm": 0.0})["norm"] > 0:
            # (a tensor whose gradient exists but is exactly zero only sees lr*wd = 3e-9 of decay: below fp32 resolution)
            assert moved, k


# bf16 gradient bounds: per-tensor error of the bf16 path's gradients against the fp32 reference, |norm(ours) - norm(ref)| / norm(ref),
# in two classes.  "gemm": convolution / linear weights and every tensor of the dense tail -- well-conditioned sums.  "bn": the BatchNorm
# affine parameters of the backbone, whose gradients are sums of ~10^6 signed terms that cancel to ~1 % of their absolute mass, so bf16
# rounding of the activations (raw, dact: 2^-9 relative each, 16 storage points along the chain) shows up amplified; stock
# torch.autocast(bfloat16) of the unmodified reference is 0.08-0.10 away from fp32 on the same tensors (tools/bf16_grad_calibration.py).
# Bounds = 2x what a B200 run printed (gpurun_out/s2, summarised in profiles/r02_parity_observations.md).
BF16_GRAD_BOUND = {"small": {"gemm": 0.10, "bn": 0.30}, "c2": {"gemm": 0.04, "bn": 0.30}}


def _bf16_grad_check(tr, c, bounds):
    gnorm = max(v["norm"] for v in c["grad_summary"].values())
    rows = []
    for k, p in tr.model.named_parameters():
        sm = c["grad_summary"].get(k)
        # skipped: tensors whose reference gradient is round-off (conv biases feeding a BatchNorm: analytically zero) or < 1e-3 of the largest
        if sm is None or sm["norm"] < 1e-3 * gnorm or synth.is_bn_fed_conv_bias(k):
            continue
        parts = k.split(".")
        cls = "bn" if parts[0] == "backbone" and parts[2] in ("1", "4") else "gemm"
        rows.append((abs(float(p.grad.double().norm()) - sm["norm"]) / sm["norm"], cls, k))
    rows.sort(reverse=True)
    worst = {cls: max([r for r in rows if r[1] == cls] or [(0.0, cls, None)]) for cls in ("gemm", "bn")}
    print(f"[bf16] case {c['name']}: worst grad-norm rel err gemm {worst['gemm'][0]:.2e} ({worst['gemm'][2]}), bn {worst['bn'][0]:.2e} ({worst['bn'][2]}); "
          "top: " + ", ".join(f"{k}={e:.3f}" for e, _, k in rows[:6]))
    for cls in ("gemm", "bn"):
        assert worst[cls][0] < bounds[cls], (cls, worst[cls])


@pytest.mark.parametrize("idx", [0, 1, 2, 3])
def test_ma_bf16_tensor_core_path(dev, gold, idx):
    """bf16 operands / fp32 accumulation (tcgen05) backbone: scores and loss within 1e-3 relative of the fp32 reference
    (north-star tolerance), identical thresholded labels; gradients within bf16 noise."""
    from cvad_b200.ma import MATrainer
    c = gold("ma.pt")["cases"][idx]
    m, noise = _ma_model(dev, c)
    tr = MATrainer(m, dev, precision="bf16")
    tr.model.train(c["train"])
    tr.model.noise = noise
    x = synth.ma_clips(c["B"], c["T"], c["H"], c["W"], c["xseed"], c["wide"]).to(dev)
    labels = c["labels"].to(dev)
    tr.optimizer.zero_grad()
    with torch.set_grad_enabled(c["train"]):
        out = tr.model(x)
        loss, comp = tr.loss_on_device(out, labels)
    e_s = rel(out["anomaly_scores"], c["anomaly_scores"], floor=1e-6)
    e_l = rel(loss, c["loss"], floor=1e-6)
    print(f"[bf16] case {c['name']}: score rel err {e_s:.2e}, loss rel err {e_l:.2e}")
    assert e_s < 1e-3 and e_l < 1e-3
    assert torch.equal(out["anomaly_scores"].cpu() > 0.5, c["anomaly_scores"] > 0.5)
    assert torch.equal(out["dense"]["det_counts"].cpu().long(), c["det_counts"])
    if c["train"]:
        loss.backward()
        _bf16_grad_check(tr, c, BF16_GRAD_BOUND["small"])


# --------------------------------------------------------------------------------------------------------- M-A0 (vad)
def _ma0_model(dev, c):
    from test_oracle_golden import ma0_eps, ma0_synth_state
    from cvad_b200.ma0 import CausalAnomalyDetector
    from cvad_b200.noise import FixedNoise
    m = CausalAnomalyDetector()
    m.load_state_dict(ma0_synth_state(c["seed"], c["margin"]), strict=True)      # same keys / shapes as vad:405-417
    return m, FixedNoise({"eps": ma0_eps(c)})


@pytest.mark.parametrize("idx", [0, 2])
def test_ma0_eval_parity_fp32(dev, gold, idx):
    """vad:419-454 forward in eval mode (fp32 path): scores, KL, adjacency, top-k detections (order, counts, dummy box) vs the reference."""
    from test_oracle_golden import ma0_input
    c = gold("ma0.pt")["cases"][idx]
    assert not c["train"]
    m, noise = _ma0_model(dev, c)
    m = m.to(dev).eval()
    m.noise = noise
    with torch.no_grad():
        out = m(ma0_input(c)[0].to(dev))
    assert set(out) >= {"anomaly_scores", "causal_factors", "adjacency_matrices", "kl_losses", "detections"}
    d = out["dense"]
    assert rel(out["anomaly_scores"], c["anomaly_scores"]) < 2e-5
    assert rel(d["kl_losses"], c["kl_losses"]) < 2e-5
    assert rel(d["adjacency_matrices"], c["adjacency"]) < 2e-5
    assert torch.equal(d["det_counts"].cpu().long(), c["det_counts"])
    assert torch.equal(d["n_tracks"].cpu().long(), c["n_tracks"])
    assert rel(d["detections"], c["detections"]) < 2e-5
    n = c["n_tracks"].tolist()
    assert len(out["causal_factors"]) == c["B"] and out["causal_factors"][0].shape == (n[0], 6)
    assert len(out["detections"][0]) == c["T"] and out["detections"][0][0].shape == (int(c["det_counts"][0, 0]), 4)
    assert len(out["kl_losses"]) == c["B"] and out["adjacency_matrices"][0].shape == (6, 6)


@pytest.mark.parametrize("idx", [1, 3])
def test_ma0_train_step_parity_fp32(dev, gold, idx):
    """vad:516-531 + backward: loss, both components, every per-tensor gradient, BN running statistics, and the parameters whose
    gradient is None in the reference (conf_head, structure_params) are not stepped."""
    from test_oracle_golden import ma0_input
    from cvad_b200.ma0 import MA0Trainer
    c = gold("ma0.pt")["cases"][idx]
    m, noise = _ma0_model(dev, c)
    tr = MA0Trainer(m, dev, precision="fp32")
    tr.model.train()
    tr.model.noise = noise
    x, labels = ma0_input(c)[0].to(dev), c["labels"].to(dev)
    tr.optimizer.zero_grad()
    out = tr.model(x)
    loss, comp = tr.loss_on_device(out, labels)
    loss.backward()
    assert rel(loss, c["loss"]) < 5e-5
    assert abs(float(comp[1]) - c["comps"]["anomaly"]) < 5e-5 * max(1.0, abs(c["comps"]["anomaly"]))
    assert abs(float(comp[2]) - c["comps"]["kl"]) < 5e-5 * max(1.0, abs(c["comps"]["kl"]))
    assert rel(out["anomaly_scores"], c["anomaly_scores"]) < 5e-5
    assert torch.equal(out["dense"]["det_counts"].cpu().long(), c["det_counts"])
    gnorm = max(v["norm"] for v in c["grad_summary"].values())
    for k, p in tr.model.named_parameters():
        sm = c["grad_summary"].get(k)
        if sm is None or sm["norm"] < 1e-5 * gnorm:
            continue
        got = float(p.grad.double().norm())
        # M-A0's only path into the backbone is the 12-column bbox head, so the backbone's BatchNorm affine gradients are ~1e-4 of the
        # largest gradient and are sums of 2*10^5 signed terms: fp32 summation order shows at the 5e-3 level there (observed 5.3e-3)
        parts = k.split(".")
        tol = 2e-2 if parts[0] == "backbone" and parts[2] in ("1", "4") else 5e-3
        assert abs(got - sm["norm"]) <= tol * sm["norm"], (k, got, sm["norm"])
        if "full" in sm:
            assert float((p.grad.cpu() - sm["full"]).double().norm()) <= tol * sm["norm"], k
    sd = tr.model.state_dict()
    for k, v in c["new_stats"].items():
        assert rel(sd[k].float(), v.float()) < 2e-5, k
    before = {k: p.detach().clone() for k, p in tr.model.named_parameters()}
    tr.optimizer.step()
    for k, p in tr.model.named_parameters():
        if not p.requires_grad:
            continue
        moved = not torch.equal(before[k], p.detach())
        if not c["has_grad"][k]:
            assert not moved, k
        elif c["grad_summary"].get(k, {"norm": 0.0})["norm"] > 0:
            assert moved, k
    assert not c["has_grad"]["detector.conf_head.weight"] and not c["has_grad"]["structure_learner.structure_params"]


@pytest.mark.parametrize("idx", [2, 3])
def test_ma0_bf16_tensor_core_path(dev, gold, idx):
    """M-A0 over the tcgen05 backbone: scores and loss within 1e-3 of the fp32 reference, identical detections and labels.  (The margin
    fixtures keep the confidences away from 0.5: with the natural near-threshold confidences of the ragged fixtures a bf16 feature error
    of 1e-2 flips anchors in and out, which is the model, not the kernels.)"""
    from test_oracle_golden import ma0_input
    from cvad_b200.ma0 import MA0Trainer
    c = gold("ma0.pt")["cases"][idx]
    m, noise = _ma0_model(dev, c)
    tr = MA0Trainer(m, dev, precision="bf16")
    tr.model.train(c["train"])
    tr.model.noise = noise
    x, labels = ma0_input(c)[0].to(dev), c["labels"].to(dev)
    tr.optimizer.zero_grad()
    with torch.set_grad_enabled(c["train"]):
        out = tr.model(x)
        loss, comp = tr.loss_on_device(out, labels)
    e_s, e_l = rel(out["anomaly_scores"], c["anomaly_scores"], floor=1e-6), rel(loss, c["loss"], floor=1e-6)
    print(f"[bf16] M-A0 case {c['name']}: score rel err {e_s:.2e}, loss rel err {e_l:.2e}")
    assert e_s < 1e-3 and e_l < 1e-3
    assert torch.equal(out["anomaly_scores"].cpu() > 0.5, c["anomaly_scores"] > 0.5)
    assert torch.equal(out["dense"]["det_counts"].cpu().long(), c["det_counts"])
    if c["train"]:
        loss.backward()
        _bf16_grad_check(tr, c, BF16_GRAD_BOUND["small"])


def test_ma0_tail_kernels_vs_oracle(dev):
    """The four M-A0 kernels against oracle/ma0.py on random inputs, values and gradients, incl. frames with 0..3 surviving anchors
    and equal confidences (anchor order must be kept)."""
    from oracle import ma0 as o
    from cvad_b200 import ma0
    g = synth.gen(91)
    B, T = 6, 7
    bbox = torch.randn(B, T, 3, 4, generator=g)
    logit = torch.randn(B, T, 3, generator=g) * 1.5
    logit[0, 0] = torch.tensor([0.7, 0.7, -1.0])          # a tie: anchors 0, 1 in that order
    logit[0, 1] = torch.tensor([-0.1, -2.0, -0.3])        # nothing passes: the dummy box
    logit[0, 2] = torch.tensor([0.2, 1.9, 0.9])           # all three, order 1, 2, 0
    conf = torch.sigmoid(logit)
    bb = bbox.clone().to(dev).requires_grad_(True)
    box, cnt, src = ma0.det_topk_decode(bb, logit.to(dev))
    w = torch.randn(B, T, 5, 4, generator=g)
    (box * w.to(dev)).sum().backward()
    bref = bbox.clone().requires_grad_(True)
    want = torch.zeros(B, T, 5, 4)
    for b in range(B):
        for t in range(T):
            order = sorted(range(3), key=lambda a: (-float(conf[b, t, a]), a))
            keep = [a for a in order if float(conf[b, t, a]) > 0.5]
            assert int(cnt[b, t]) == max(len(keep), 1)
            assert src[b, t, :len(keep)].tolist() == keep and (len(keep) > 0 or int(src[b, t, 0]) == -1)
    want_box = torch.stack([torch.stack([torch.cat([bref[b, t, [a for a in sorted(range(3), key=lambda a: (-float(conf[b, t, a]), a))
                                                                 if float(conf[b, t, a]) > 0.5]],
                                                    torch.zeros(5, 4)])[:5] for t in range(T)]) for b in range(B)])
    (want_box * w).sum().backward()
    assert torch.equal(box.detach().cpu(), want_box.detach())
    assert torch.equal(bb.grad.cpu(), bref.grad)
    assert src[0, 0, :2].tolist() == [0, 1] and int(cnt[0, 1]) == 1 and src[0, 2, :3].tolist() == [1, 2, 0]
    # per-track score rows + masked mean + loss
    z = torch.randn(B, 5, 6, generator=g)
    pr = torch.randn(B, 5, 6, generator=g)
    pr[0, 0, 0] = z[0, 0, 0]                              # |.| at zero: sign(0) = 0 like torch.abs
    ntr = torch.tensor([1, 2, 3, 5, 4, 1], dtype=torch.int32)
    kl = torch.randn(B, generator=g).abs()
    kl[3] = float("inf")
    labels = torch.tensor([0, 1, 1, 0, 1, 0])
    zd, pd = z.clone().to(dev).requires_grad_(True), pr.clone().to(dev).requires_grad_(True)
    kd = kl.clone().to(dev).requires_grad_(True)
    rows = ma0.score_rows(zd, pd)
    s = torch.sigmoid(rows.sum(-1))
    sc = ma0.masked_mean(s, ntr.to(dev))
    loss, comp = ma0.ma0_loss(sc, kd, labels.to(dev))
    loss.backward()
    zr, prr, kr = z.clone().requires_grad_(True), pr.clone().requires_grad_(True), kl.clone().requires_grad_(True)
    rows_r = torch.cat([zr, prr, (zr - prr).abs()], -1)
    ok = (torch.arange(5).view(1, -1) < ntr.view(-1, 1)).float()
    sc_r = (torch.sigmoid(rows_r.sum(-1)) * ok).sum(1) / ntr
    lr, cr = o.ma0_loss({"anomaly_scores": sc_r, "kl_losses": kr}, labels)
    lr.backward()
    assert rel(rows, rows_r) < 1e-6 and rel(sc, sc_r) < 1e-6 and rel(loss, lr) < 1e-6
    assert abs(float(comp[1]) - cr["anomaly"]) < 1e-6 and abs(float(comp[2]) - cr["kl"]) < 1e-6
    assert rel(zd.grad, zr.grad, floor=1e-6) < 1e-5 and rel(pd.grad, prr.grad, floor=1e-6) < 1e-5
    assert rel(kd.grad, kr.grad, floor=1e-9) < 1e-6 and float(kd.grad[3]) == 0.0
    # no finite KL term at all: the KL part is 0 (vad:522) and carries no gradient
    kinf = torch.full((B,), float("nan"), device=dev, requires_grad=True)
    l2, c2 = ma0.ma0_loss(sc.detach(), kinf, labels.to(dev))
    l2.backward()
    assert float(c2[2]) == 0.0 and float(kinf.grad.abs().max()) == 0.0 and rel(l2, c2[1]) < 1e-7


@pytest.mark.parametrize("kind", ["ma0", "ma"])
def test_streaming_window_scorer_equals_clip_by_clip(dev, gold, kind):
    """Sliding windows over a frame stream (stride 4, 16-frame clips): every frame's backbone pass is computed once, when it arrives, and the
    window scores equal scoring each window as its own clip -- against the unmodified reference for M-A0 (tests/golden/ma0.pt 'stream')
    and against the model's own clip forward for M-A.  Frames are pushed in uneven chunks so that the ring wraps."""
    from test_oracle_golden import ma0_input, ma_noise, ma_synth_state
    from cvad_b200.ma0 import StreamingWindowScorer
    from cvad_b200.noise import FixedNoise
    c = [k for k in gold("ma0.pt")["cases"] if k.get("stream")][0]
    clips, seq = ma0_input(c)
    B, T = c["B"], c["T"]
    if kind == "ma0":
        m, _ = _ma0_model(dev, c)
        want = c["anomaly_scores"]
    else:
        from cvad_b200.ma import CausalAnomalyDetector
        m = CausalAnomalyDetector()
        m.load_state_dict(ma_synth_state(4, True), strict=True)
        want = None
    m = m.to(dev).eval()
    eps = torch.randn(B, 5, 6, generator=synth.gen(c["xseed"] + 1))
    if want is None:
        m.noise = FixedNoise({"eps": eps})
        with torch.no_grad():
            want = m(clips.to(dev))["anomaly_scores"].cpu()
    sc = StreamingWindowScorer(m, clip_len=T, stride=4, capacity=24)
    got, first = [], []
    pos = 0
    for n in (5, 8, 3, 7, 1, 4):                     # 28 frames = 16 + 4*3; capacity 24 < 28: the ring wraps
        chunk = seq[pos:pos + n].to(dev)
        pos += n
        done = (max(pos - T, -1) // 4 + 1 if pos >= T else 0) - len(got)
        m.noise = FixedNoise({"eps": eps[len(got):len(got) + done]}) if done > 0 else m.noise
        s, w0 = sc.push(chunk)
        assert s.shape[0] == done and w0 == len(got)
        got += s.cpu().tolist()
    assert pos == seq.shape[0] and len(got) == B
    assert rel(torch.tensor(got), want) < 2e-5, (got, want)


# ---- the BENCHMARKED shape: 32 clips x 16 frames x 240 x 360 (BASELINE.json configs[1]); every tcgen05 template instance sees the
# same number of work items per CTA as in bench.py (tests/golden/ma_c2.pt comes from the unmodified reference, tools/make_golden.py)
RANK_TIE_EPS = 2e-3      # relative to the largest score: two clips closer than this may swap ranks under the 1e-3 score tolerance


def _same_ranking(got, want, tie_eps):
    """Every pair of clips that the reference separates by more than tie_eps * max|score| is ordered identically."""
    got, want = got.double().cpu(), want.double().cpu()
    dw = want.unsqueeze(0) - want.unsqueeze(1)
    dg = got.unsqueeze(0) - got.unsqueeze(1)
    decided = dw.abs() > tie_eps * float(want.abs().max())
    return bool((torch.sign(dw)[decided] == torch.sign(dg)[decided]).all()), int(decided.sum()) // 2


def _c2_step(dev, c, precision):
    from cvad_b200.ma import MATrainer
    m, noise = _ma_model(dev, c)
    tr = MATrainer(m, dev, precision=precision)
    tr.model.train()
    tr.model.noise = noise
    x = synth.ma_clips(c["B"], c["T"], c["H"], c["W"], c["xseed"], c["wide"]).to(dev)
    labels = c["labels"].to(dev)
    tr.optimizer.zero_grad()
    out = tr.model(x)
    loss, comp = tr.loss_on_device(out, labels)
    loss.backward()
    torch.cuda.synchronize()
    return tr, out, loss, comp


@pytest.mark.parametrize("idx", [0, 1])
def test_ma_c2_benchmarked_shape_fp32(dev, gold, idx):
    """cad:637-688 at 512 frames, fp32 mode: loss + 4 components, scores, per-tensor gradients, BN running statistics (5e-5 / 5e-3)."""
    c = gold("ma_c2.pt")["cases"][idx]
    tr, out, loss, comp = _c2_step(dev, c, "fp32")
    assert rel(loss, c["loss"]) < 5e-5
    for i, k in enumerate(("classification", "anomaly", "causal", "kl")):
        assert abs(float(comp[i + 1]) - c["comps"][k]) < 5e-5 * max(1.0, abs(c["comps"][k])), k
    assert rel(out["anomaly_scores"], c["anomaly_scores"]) < 5e-5
    assert rel(out["direct_predictions"], c["direct_predictions"]) < 5e-5
    assert rel(out["dense"]["kl_losses"], c["kl_losses"]) < 5e-5
    assert torch.equal(out["dense"]["n_tracks"].cpu().long(), c["n_tracks"])
    gnorm = max(v["norm"] for v in c["grad_summary"].values())
    for k, p in tr.model.named_parameters():
        sm = c["grad_summary"].get(k)
        if sm is None or sm["norm"] < 1e-5 * gnorm:
            continue
        got = float(p.grad.double().norm())
        assert abs(got - sm["norm"]) <= 5e-3 * sm["norm"], (k, got, sm["norm"])
        if "full" in sm:
            assert float((p.grad.cpu() - sm["full"]).double().norm()) <= 5e-3 * sm["norm"], k
    sd = tr.model.state_dict()
    for k, v in c["new_stats"].items():
        assert rel(sd[k].float(), v.float()) < 2e-5, k


@pytest.mark.parametrize("idx", [0, 1])
def test_ma_c2_benchmarked_shape_bf16(dev, gold, idx):
    """The benchmarked configuration itself (bf16 operands, tcgen05, 512 frames): scores and loss within 1e-3 of the fp32 reference,
    identical thresholded labels (0.5 and the p95 threshold of s1:60) and identical ranking up to the stated tie epsilon."""
    import numpy as np
    c = gold("ma_c2.pt")["cases"][idx]
    tr, out, loss, comp = _c2_step(dev, c, "bf16")
    got, want = out["anomaly_scores"].detach().cpu(), c["anomaly_scores"]
    e_s, e_l = rel(got, want, floor=1e-6), rel(loss, c["loss"], floor=1e-6)
    same, pairs = _same_ranking(got, want, RANK_TIE_EPS)
    print(f"[bf16 C2] case {c['name']}: score rel err {e_s:.2e}, loss rel err {e_l:.2e}, {pairs} decided pairs ranked identically: {same}")
    assert e_s < 1e-3 and e_l < 1e-3
    for i, k in enumerate(("classification", "anomaly", "causal", "kl")):
        assert abs(float(comp[i + 1]) - c["comps"][k]) < 1e-3 * max(1.0, abs(c["comps"][k])), k
    assert rel(out["direct_predictions"], c["direct_predictions"]) < 1e-3
    assert torch.equal(got > 0.5, want > 0.5)
    thr = float(np.percentile(want.numpy(), 95))
    clear = (want - thr).abs() > RANK_TIE_EPS * float(want.abs().max())
    assert torch.equal((got > thr)[clear], (want > thr)[clear])
    assert same
    # detections are hard window tests on continuous box coordinates (cad:217-218): a box within bf16 noise of a window edge may flip, so
    # the per-frame counts are compared as a mismatch rate (observed: 3 of 512 frames with the live detector, 0 with the stock one); the
    # per-clip track counts -- what the causal branch consumes -- must agree
    dc = out["dense"]["det_counts"].cpu().long()
    flips = int((dc != c["det_counts"]).sum())
    print(f"[bf16 C2] case {c['name']}: {flips} of {dc.numel()} per-frame detection counts differ from the fp32 reference")
    assert flips <= 0.02 * dc.numel()
    assert torch.equal(out["dense"]["n_tracks"].cpu().long(), c["n_tracks"])
    _bf16_grad_check(tr, c, BF16_GRAD_BOUND["c2"])
    sd = tr.model.state_dict()
    for k, v in c["new_stats"].items():
        if "bn1" not in k:          # the frozen stem's statistics come from the tf32 stem (tested in test_flat_gpu.py)
            assert rel(sd[k].float(), v.float()) < 5e-3, k



@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_ma_uint8_frames_equal_host_normalised_frames(dev, precision):
    """SURVEY 8(f1) / K1: raw uint8 grayscale frames (cad:89-96) normalised on the device give bit-identical scores to the reference's
    host-side Normalize(0.5, 0.5) (cad:1177-1179) -- the input crosses PCIe at 1 byte per pixel instead of 4."""
    from test_oracle_golden import ma_synth_state
    from cvad_b200.ma import CausalAnomalyDetector
    from cvad_b200.noise import FixedNoise
    B, T, H, W = 3, 4, 120, 180
    u8 = torch.randint(0, 256, (B, T, 1, H, W), generator=synth.gen(5), dtype=torch.uint8)
    xf = (u8.float() - 0.5) / 0.5
    m = CausalAnomalyDetector()
    m.load_state_dict(ma_synth_state(4, True), strict=True)
    m = m.to(dev).eval().set_precision(precision)
    eps = torch.randn(B, 5, 6, generator=synth.gen(6))
    outs = []
    for x in (xf, u8):
        m.noise = FixedNoise({"eps": eps})
        with torch.no_grad():
            outs.append(m(x.to(dev)))
    # the claim is about the input path: the backbone's features are bit-identical.  The dense tail sums its split-K GEMMs with red.add
    # (and runs its independent branches concurrently), so the last bits of the scores depend on the order the partial sums arrive in
    assert torch.equal(outs[0]["dense"]["features"], outs[1]["dense"]["features"])
    assert rel(outs[0]["anomaly_scores"], outs[1]["anomaly_scores"], floor=1e-6) < 1e-5


# 3 optimizer steps against the reference's own train_model loop (cad:609-709: AdamW 3e-4 / 1e-5, clip_grad_norm_ 1.0, frozen stem).
# Distance measure: |ours - ref|_2 / |ref - start|_2 per tensor on a strided sample.  Adam's first steps move every element by ~lr
# whatever its gradient's size, so elements whose gradient is round-off-sized differ by O(lr) between ANY two summation orders: the
# oracle (fp32, CPU) is already 0.10 away from the reference by this measure (tools/make_golden.py prints it).
# bf16: the BatchNorm affine gradients carry ~10 % noise (see BF16_GRAD_BOUND) and Adam normalises every element's step to ~lr, so after three
# steps those 32..256-element vectors sit most of a step-length away; the bound there only says "same order of motion".
TRAJ_BOUND = {"fp32": {"gemm": 0.4, "bn": 0.4, "stat": 3e-3}, "bf16": {"gemm": 0.8, "bn": 1.5, "stat": 6e-2}}


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name", ["traj_sat", "traj_live"])
def test_ma_trajectory_vs_reference_train_model(dev, gold, name, precision):
    from test_oracle_golden import ma_synth_state
    from cvad_b200.ma import CausalAnomalyDetector, MATrainer
    from cvad_b200.noise import FixedNoise
    g = gold("ma_traj.pt")[name]
    B, T = g["B"], g["T"]
    P0 = ma_synth_state(g["seed"], g["live"])
    m = CausalAnomalyDetector()
    m.load_state_dict(P0, strict=True)
    tr = MATrainer(m, dev, num_epochs=1, lr=3e-4, precision=precision)
    tr.model.train()
    losses = []
    for xs in g["xseeds"]:
        x = synth.ma_clips(B, T, g["H"], g["W"], xs, g["wide"]).to(dev)
        y = (torch.rand(B, generator=synth.gen(xs + 9)) < 0.5).long().to(dev)
        eps = torch.randn(B, 5, 6, generator=synth.gen(xs + 1))
        keep = {"det0": synth.keep_mask((B, T, 512), 0.3, xs + 2), "det1": synth.keep_mask((B, T, 256), 0.2, xs + 3),
                "scorer0": synth.keep_mask((B, 64), 0.2, xs + 4), "cls0": synth.keep_mask((B, 512), 0.3, xs + 5),
                "cls1": synth.keep_mask((B, 256), 0.2, xs + 6)}
        tr.model.noise = FixedNoise({"eps": eps, **keep})
        comp, _ = tr.train_step(x, y)
        losses.append(float(comp[0]))
    # Step 1 starts from identical parameters: the north-star tolerance applies (5e-5 fp32 / 1e-3 bf16).  From step 2 on the parameters
    # themselves differ: Adam's first updates are lr * g / |g| per element, so an element whose gradient is at round-off level moves by a
    # full +-lr with a sign that depends on the summation order (the reference's own CPU run vs the fp32 oracle already differ that way),
    # and the loss inherits it -- the bound grows per step (observed on a B200: fp32 3e-6 / 3e-4, bf16 5e-4 / 3e-3 at steps 2 / 3).
    tol = {"fp32": (5e-5, 2e-4, 1e-3), "bf16": (1e-3, 2e-3, 1e-2)}[precision]
    errs = [abs(a - b) / abs(b) for a, b in zip(losses, g["oracle_losses"])]
    print(f"[traj {name} {precision}] losses {losses} (reference-pinned oracle {g['oracle_losses']}), rel err {[f'{e:.1e}' for e in errs]}")
    sd = tr.model.state_dict()

    def sample(t):              # the fixture keeps at most sample_cap elements of each tensor's strided sample
        return synth.strided_sample(synth.strided_sample(t), g["sample_cap"])
    worst, worst_stat = {"gemm": (0.0, None), "bn": (0.0, None)}, 0.0
    for k, ref in g["final_sample"].items():
        got = sample(sd[k].float().cpu())
        start = sample(P0[k].float())
        moved = float((ref - start).double().norm())
        d = float((got - ref).double().norm())
        if "running" in k:
            if not ("bn1" in k and precision == "bf16"):       # the frozen stem's statistics come from the tf32 stem (test_flat_gpu.py)
                worst_stat = max(worst_stat, d / float(ref.double().norm()))
            continue
        if synth.is_bn_fed_conv_bias(k):
            continue            # reference: Adam-amplified round-off (analytically zero gradient); here: exactly zero gradient
        if moved == 0.0:
            assert d == 0.0, k   # frozen stem, saturated detector / structure learner: untouched (not even weight decay)
            continue
        parts = k.split(".")
        cls = "bn" if parts[0] == "backbone" and parts[2] in ("1", "4") else "gemm"
        if d / moved > worst[cls][0]:
            worst[cls] = (d / moved, k)
    print(f"[traj {name} {precision}] worst |ours - ref| / |ref - start|: gemm-class {worst['gemm'][0]:.3f} ({worst['gemm'][1]}), "
          f"BatchNorm affine {worst['bn'][0]:.3f} ({worst['bn'][1]}); worst running-statistic rel err {worst_stat:.1e}")
    for e, t in zip(errs, tol):
        assert e <= t, (errs, tol)
    assert abs(sum(losses) / 3 - g["mean_loss"]) <= tol[2] * abs(g["mean_loss"])
    assert worst_stat < TRAJ_BOUND[precision]["stat"]
    assert worst["gemm"][0] < TRAJ_BOUND[precision]["gemm"] and worst["bn"][0] < TRAJ_BOUND[precision]["bn"], worst


# --------------------------------------------------------------------------------------------------------- M-D
def _md_model(dev, c):
    from cvad_b200.md import VideoAutoEncoder
    from test_oracle_golden import md_reference_order, md_state_like, md_synth_state
    m = VideoAutoEncoder()
    assert list(m.state_dict().keys()) == c["state_keys"]          # same names, same order as the reference module
    m.load_state_dict(md_state_like(md_reference_order(md_synth_state(c["seed"]), c["state_keys"]), c["seed"]), strict=True)
    return m.to(dev)


@pytest.mark.parametrize("idx", [0, 1])
def test_md_eval_parity(dev, gold, idx):
    """a19-a20: reconstruction, LSTM sequence feature, memory score and the combined clip score (cad1:545-552), fp32."""
    from cvad_b200 import md
    c = gold("md.pt")["cases"][idx]
    assert not c["train"]
    m = _md_model(dev, c).eval()
    x = synth.md_clips(c["B"], c["T"], seed=c["xseed"])
    with torch.no_grad():
        out = m(x.to(dev))
    assert out["reconstructed"].shape == (c["B"], c["T"], 1, 64, 64)
    assert rel(out["reconstructed"][:, 0], c["recon_frame0"]) < 2e-5 and rel(out["reconstructed"][:, -1], c["recon_frame0"]) < 2e-5
    assert rel(out["sequence_feature"], c["sequence_feature"]) < 2e-5
    assert rel(out["frame_features"], c["frame_features"]) < 2e-5
    assert rel(out["anomaly_score"], c["anomaly_score"], floor=1e-6) < 2e-5
    scores, labels, recons, mems = md.calculate_anomaly_scores(m, [(x, torch.zeros(c["B"]))], device=dev)
    assert rel(torch.tensor(scores), c["combined"]) < 2e-5 and labels.shape == (c["B"],)


@pytest.mark.parametrize("idx", [2, 3])
def test_md_train_step_parity(dev, gold, idx):
    """Reconstruction loss, every parameter gradient, T sequential BN running-stat updates, memory-bank update (cad1:380-425)."""
    from cvad_b200.md import MDTrainer
    c = gold("md.pt")["cases"][idx]
    assert c["train"]
    tr = MDTrainer(_md_model(dev, c), dev)
    tr.model.train()
    x = synth.md_clips(c["B"], c["T"], seed=c["xseed"]).to(dev)
    tr.optimizer.zero_grad()
    out = tr.model(x)
    from cvad_b200.md import reconstruction_loss
    loss = reconstruction_loss(x, out["reconstructed"])
    tr.model.update_memory(out["sequence_feature"])
    loss.backward()
    assert abs(float(loss) - c["loss"]) < 2e-5 * max(1.0, abs(c["loss"]))
    gmax = max(v["norm"] for v in c["grads"].values())
    for k, p in tr.model.named_parameters():
        gs = c["grads"][k]
        # per-time-step BatchNorm over 32..96 values amplifies fp32 round-off (the reference and its own restatement differ by ~1e-3)
        assert abs(float(p.grad.double().norm()) - gs["norm"]) <= 5e-3 * gmax, (k, float(p.grad.norm()), gs["norm"])
        if gs["full"] is not None and gs["norm"] > 1e-2 * gmax:
            assert float((p.grad.cpu() - gs["full"]).double().norm()) <= 2e-2 * gs["norm"] + 1e-3 * gmax, k
    sd = tr.model.state_dict()
    for k, v in c["new_stats"].items():
        assert rel(sd[k].float(), v.float(), floor=1e-6) < 5e-5, k
    assert rel(sd["normal_memory"][37:37 + c["B"]], c["memory_rows"]) < 2e-5
    before = tr.model.encoder[13].weight.detach().clone()
    tr.optimizer.step()
    assert not torch.equal(before, tr.model.encoder[13].weight.detach())


@pytest.mark.parametrize("N,T", [(3, 5), (7, 1), (2, 16)])
def test_lstm_kernel_vs_torch(dev, N, T):
    from cvad_b200 import ops
    lstm = torch.nn.LSTM(64, 64, batch_first=True)           # plain fp32 reference on the CPU (cuDNN's RNN may use TF32)
    x = torch.randn(N, T, 64, requires_grad=True)
    _, (h, _) = lstm(x)
    gy = torch.randn(N, 64)
    gr = torch.autograd.grad(h[-1], [x, lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0], gy)
    gy = gy.to(dev)
    x2 = x.detach().clone().to(dev).requires_grad_(True)
    ps = [p.detach().clone().to(dev).requires_grad_(True) for p in (lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0)]
    gi = ops.linear_act(x2.reshape(N * T, 64), ps[0], ps[2]).reshape(N, T, 256)
    hT = ops.lstm_last(gi, ps[1], ps[3])
    assert rel(hT, h[-1]) < 1e-5
    hT.backward(gy)
    assert rel(x2.grad, gr[0]) < 1e-4
    for p, g in zip(ps, gr[1:]):
        assert rel(p.grad, g) < 1e-4


def test_conv_transpose_and_memory_score_vs_torch(dev):
    import torch.nn.functional as F
    from cvad_b200 import ops
    torch.backends.cudnn.allow_tf32 = False          # the torch reference must be plain fp32
    torch.backends.cuda.matmul.allow_tf32 = False
    x = torch.randn(3, 16, 5, 7, device=dev, requires_grad=True)
    w = (torch.randn(16, 8, 4, 4, device=dev) * 0.1).requires_grad_(True)
    b = torch.randn(8, device=dev, requires_grad=True)
    ref = torch.sigmoid(F.conv_transpose2d(x, w, b, stride=2, padding=1))
    gy = torch.randn_like(ref)
    gr = torch.autograd.grad(ref, (x, w, b), gy)
    x2, w2, b2 = (t.detach().clone().requires_grad_(True) for t in (x, w, b))
    y = ops.channel_bias_act(ops.conv_transpose2d(x2, w2, 2, 1), b2, ops.ACT_SIGMOID)
    assert y.shape == ref.shape and rel(y, ref) < 1e-5
    y.backward(gy)
    assert rel(x2.grad, gr[0]) < 1e-4 and rel(w2.grad, gr[1]) < 1e-4 and rel(b2.grad, gr[2]) < 1e-4
    seq, mem = torch.randn(5, 64, device=dev), torch.randn(500, 64, device=dev)
    zn, mn = F.normalize(seq, dim=-1), F.normalize(mem[:123], dim=-1)
    want = (1 - (zn @ mn.t()).clamp(-1, 1)).min(dim=1)[0].clamp(0, 2) / 2
    assert rel(ops.memory_score(seq, mem, 123), want, floor=1e-6) < 1e-5
    assert float(ops.memory_score(seq, mem, 9).abs().max()) == 0.0


# --------------------------------------------------------------------------------------------------------- M-E / windows / pseudo-labels
def test_me_forward_and_sliding_windows(dev, gold):
    """a21: the visualiser's model (bbox:51-101) on a batch, and all stride-4 windows of a video scored in one batch
    (bbox:392-415 scores them one batch-1 forward at a time) -- same scores, same adjacency."""
    from cvad_b200 import me
    g = gold("me.pt")
    m = me.CausalAnomalyDetector()
    assert list(m.state_dict().keys()) == g["state_keys"]
    m.load_state_dict(synth.synth_fill(m.state_dict(), 555), strict=True)
    m = m.to(dev).eval()
    x = synth.mb_clips(4, 8, 64, 64, 77)
    with torch.no_grad():
        s, a, f = m(x.to(dev))
    assert s.shape == (4,) and a.shape == (4, 16, 16) and f.shape == (4, 1024)
    assert rel(s, g["scores"]) < 2e-5 and rel(a, g["adj"]) < 2e-5 and rel(f, g["feat"]) < 2e-5
    frames = torch.rand(41, 3, 64, 64, generator=synth.gen(78))
    starts, scores, adjs, feats = me.score_windows(m, frames, device=dev)
    assert list(starts) == list(range(0, 41 - 8, 4))
    assert rel(torch.tensor(scores), g["win_scores"]) < 2e-5 and rel(torch.tensor(adjs), g["win_adj"]) < 2e-5
    one = me.predict_anomaly_for_clip(m, frames[4:12].permute(1, 0, 2, 3).numpy(), device=dev)
    assert abs(one[0] - float(g["win_scores"][1])) < 2e-5 and one[1].shape == (16, 16)
    recs = me.extract_anomalous_windows(m, frames, threshold=float(g["win_scores"].median()), device=dev)
    assert len(recs) == int((g["win_scores"] > g["win_scores"].median()).sum()) and all(r["end_frame"] - r["start_frame"] == 8 for r in recs)


def test_create_unsupervised_labels(dev, gold):
    """a22 (s1:36-67): p95 threshold over all scores of a loader."""
    import numpy as np
    from cvad_b200.mb import MiniCausalVAD, create_unsupervised_labels
    tr = MiniCausalVAD(device=dev)
    tr.model.load_state_dict(gold("best_improved_model.pth")["model_state_dict"], strict=True)
    loader = [(synth.mb_clips_bright(4, 8, 64, 64, 500 + i), torch.zeros(4)) for i in range(6)]
    scores, labels, thr = create_unsupervised_labels(loader, tr, 95)
    assert scores.shape == (24,) and labels.shape == (24,)
    assert abs(thr - np.percentile(scores, 95)) < 1e-12 and int(labels.sum()) == int((scores > thr).sum()) >= 1
    ref = torch.cat([tr.model(v.to(dev))[0].reshape(-1) for v, _ in loader]).detach().cpu().numpy()
    assert np.allclose(scores, ref, rtol=0, atol=1e-7)


# --------------------------------------------------------------------------------------------------------- long-sequence sweep
@pytest.mark.parametrize("T", [64, 128, 256])
def test_long_sequence_inference_sweep_sharded(dev, gold, T):
    """BASELINE config 5: clip scoring at 64-256 frames per clip, clips sharded over 2/4/8 ranks with no communication.  The CUDA
    path must equal the CPU oracle on the whole batch (fp32, 1e-5), and every rank's shard (DataParallel.shard) must reproduce its
    slice of the unsharded result bit for bit -- eval-mode BatchNorm, no cross-clip coupling."""
    from oracle import mb as o_mb, mc as o_mc
    from cvad_b200.mb import CausalAnomalyDetector as MB
    from cvad_b200.mc import SimpleVideoAnomalyDetector
    from cvad_b200.parallel import DataParallel
    B = 8
    g = gold("mc.pt")
    mc = SimpleVideoAnomalyDetector().to(dev).eval()
    mc.load_state_dict(_mc_synth(g), strict=True)
    P = {k: v.detach().cpu() for k, v in mc.state_dict().items()}
    x = synth.mc_clips(B, T, 64, 64, 900 + T)
    with torch.no_grad():
        full = mc(x.to(dev))
    assert rel(full, o_mc.mc_forward(P, x), floor=1e-6) < 1e-5
    mbm = MB().to(dev).eval()
    Pb = {k: v.detach().cpu() for k, v in mbm.state_dict().items()}
    xb = synth.mb_clips(B, T, 64, 64, 700 + T)
    with torch.no_grad():
        sb, ab, fb = mbm(xb.to(dev))
    so, ao, fo = o_mb.mb_forward(Pb, xb)
    assert rel(sb, so, floor=1e-6) < 1e-5 and rel(ab, ao) < 1e-5 and rel(fb, fo) < 1e-5
    for world in (2, 4, 8):
        parts = []
        for rank in range(world):
            dp = DataParallel.__new__(DataParallel)          # shard arithmetic only: no process group on a single GPU
            dp.world, dp.rank = world, rank
            lo, hi = dp.shard(B)
            with torch.no_grad():
                parts.append(mc(x[lo:hi].to(dev)))
        assert rel(torch.cat(parts), full, floor=1e-6) < 1e-6          # split-K of the dense layers depends on the batch size


# --------------------------------------------------------------------------------------------------------- CUDA-graph step
@pytest.mark.parametrize("split", [False, True])
def test_graphed_train_step_matches_eager(dev, split):
    """One CUDA graph per step (graphs.GraphedStep): building it must not advance training, replays must equal eager steps, and a
    scheduler's LR change must reach the captured optimizer kernel through the device-side LR.  ``split`` = the data-parallel
    form: graph(zero_grad..backward) -> eager hook (the NCCL all-reduce; here an identity op on the arena) -> graph(clip+AdamW)."""
    from cvad_b200.ma import CausalAnomalyDetector, MATrainer
    from cvad_b200.noise import FixedNoise
    B, T, H, W = 2, 4, 64, 96

    def make():
        torch.manual_seed(7)
        tr = MATrainer(CausalAnomalyDetector(), dev, precision="bf16")
        tr.model.train()
        g = synth.gen(11)
        noise = {"eps": torch.randn(B, 5, 6, generator=g), "det0": synth.keep_mask((B, T, 512), 0.3, 1),
                 "det1": synth.keep_mask((B, T, 256), 0.2, 2), "scorer0": synth.keep_mask((B, 64), 0.2, 3),
                 "cls0": synth.keep_mask((B, 512), 0.3, 4), "cls1": synth.keep_mask((B, 256), 0.2, 5)}
        tr.model.noise = FixedNoise({k: v.to(dev) for k, v in noise.items()})       # device-resident: replayable inside a graph
        return tr

    xs = [synth.ma_clips(B, T, H, W, 20 + i, wide=False).to(dev) for i in range(3)]
    ys = [torch.tensor([0, 1], device=dev), torch.tensor([1, 1], device=dev), torch.tensor([0, 0], device=dev)]
    eager, eager2, graphed = make(), make(), make()
    p0 = graphed.optimizer.arena.p.clone()
    if split:
        hook_calls = [0]

        def hook(arena):
            hook_calls[0] += 1
            arena.g.mul_(1.0)
        graphed.optimizer.pre_step_hook = hook
    gs = graphed.graphed_train_step(xs[0], ys[0])
    assert len(gs.stages) == (1 if split else 0)
    assert torch.equal(graphed.optimizer.arena.p, p0), "capturing the graph must not change the parameters"
    assert gs.launches > 50
    for i in range(3):
        if i == 2:                      # an LR scheduler step between replays
            for tr in (eager, eager2, graphed):
                tr.optimizer.param_groups[0]["lr"] = 1e-3
        ce, _ = eager.train_step(xs[i], ys[i])
        eager2.train_step(xs[i], ys[i])
        cg, _ = gs(xs[i], ys[i])
        # step 0 starts from identical parameters: the losses agree to round-off.  Later steps start from parameters that Adam's sign
        # amplification of round-off-sized gradients has already spread (see below; observed 3e-3 at the third step, after the LR change)
        assert rel(cg, ce, floor=1e-6) < (1e-4 if i == 0 else 1e-2), (i, cg, ce)
        if i == 0:
            # after ONE step the first-moment buffer is 0.1 x the gradient taken at identical parameters: linear in the gradient, so
            # graph and eager must agree to round-off (later steps inherit Adam's sign amplification, see below)
            m_err = rel(graphed.optimizer.arena.m, eager.optimizer.arena.m, floor=1e-12)
            print(f"[graph] first-step moment buffers: graph-vs-eager {m_err:.3e}")
            assert m_err < 3e-2
    if split:
        assert hook_calls[0] == 3 + 3, hook_calls       # 3 warm-up executions + one eager call per replay, none at capture
    pe, pe2, pg = eager.optimizer.arena.p, eager2.optimizer.arena.p, graphed.optimizer.arena.p
    moved = float((pe - p0).abs().mean())
    noise = float((pe - pe2).abs().mean())         # run-to-run spread of two EAGER runs (Adam amplifies atomics round-off)
    diff = float((pe - pg).abs().mean())
    print(f"[graph] mean |dp| {moved:.3e}, eager-vs-eager {noise:.3e}, graph-vs-eager {diff:.3e}")
    assert moved > 1e-4
    # Adam turns the sign of a round-off-sized gradient into a full +-lr move and the order of the kernels' fp32 atomics differs from
    # run to run (two eager runs can also happen to be bit-identical), so parameters are compared loosely after three steps
    assert diff <= 3 * noise + 0.4 * moved          # observed 0.1-0.27 x moved (two eager runs can be bit-identical: noise = 0)
    # the third step ran at lr 1e-3 in all three: had the graph kept the captured 3e-4 it would trail by ~0.7e-3 per parameter
    last = float(((pg - p0).abs().mean()))
    assert abs(last - moved) < 0.1 * moved


# --------------------------------------------------------------------------------------------------------- driver: resume + history (8(f4))
def test_train_driver_resume_matches_uninterrupted_run(dev, tmp_path):
    """s2:339-468 driver: history JSON schema, checkpoint dict keys (s2:437-455), and an actual resume -- a run interrupted after epoch 2
    and resumed from checkpoint_epoch_1.pth (model, AdamW moments + step counters, scheduler, history, best score, device RNG) ends where
    the uninterrupted 4-epoch run ends (weight-gradient atomics make the two runs equal to ~1e-6, not bitwise)."""
    import json
    from cvad_b200 import train as drv
    import avenue_dataset_usage as a

    def loaders():
        return a.create_avenue_dataloaders("synthetic:16", batch_size=4, clip_length=8, frame_size=(64, 64))

    class Killed(Exception):
        pass

    def kill_after_epoch_1(epoch, _hist):
        if epoch == 1:
            raise Killed()

    def run(out, resume=None, hook=None):
        torch.manual_seed(77)
        torch.cuda.manual_seed(77)
        return drv.train_improved_minicausal_vad("synthetic:16", num_epochs=4, batch_size=4, save_interval=1, output_dir=out, resume=resume,
                                                 device=dev, loaders=loaders(), verbose=False, on_epoch_end=hook)

    full, hist_full = run(tmp_path / "full")
    with pytest.raises(Killed):
        run(tmp_path / "part", hook=kill_after_epoch_1)           # the same 4-epoch job, killed after its second epoch
    ck = torch.load(tmp_path / "part" / "checkpoint_epoch_1.pth", map_location="cpu", weights_only=False)
    assert {"model_state_dict", "optimizer_state_dict", "scheduler_state_dict", "epoch", "training_history"} <= set(ck) and ck["epoch"] == 1
    best = torch.load(tmp_path / "part" / "best_improved_model.pth", map_location="cpu", weights_only=False)
    assert set(best) == {"model_state_dict", "optimizer_state_dict", "epoch", "eval_metrics"}
    resumed, hist_res = run(tmp_path / "part", resume=tmp_path / "part" / "checkpoint_epoch_1.pth")
    assert hist_res["epochs"] == [1, 2, 3, 4] == hist_full["epochs"] and len(hist_res["train_losses"]) == 4
    for k in ("train_losses", "learning_rates"):
        assert np.allclose(hist_res[k], hist_full[k], rtol=1e-4, atol=1e-7), (k, hist_res[k], hist_full[k])
    for (k, v), (_, w) in zip(full.model.state_dict().items(), resumed.model.state_dict().items()):
        assert float((v - w).abs().max()) <= 1e-4 * max(float(v.abs().max()), 1e-3), k
    on_disk = json.load(open(tmp_path / "part" / "improved_training_history.json"))
    assert set(on_disk) == {"train_losses", "loss_components", "evaluation_metrics", "epochs", "learning_rates"}
    assert len(on_disk["evaluation_metrics"]) == len(hist_res["evaluation_metrics"]) and set(on_disk["evaluation_metrics"][0]) == {
        "mean_score", "std_score", "min_score", "max_score", "score_range", "avg_edges", "avg_sparsity", "unique_graphs"}
    assert set(on_disk["loss_components"][0]) == {"anomaly_loss", "acyclicity_loss", "sparsity_loss", "consistency_loss", "structure_loss",
                                                  "edge_count", "sparsity_ratio"}
