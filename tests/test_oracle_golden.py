"""The oracle restatement (oracle/) against the committed golden fixtures produced by the reference itself
(tools/make_golden.py).  Runs on CPU; pins the oracle without needing /root/reference."""
import os

import pytest
import torch

import synth
from oracle import ma as o_ma
from oracle import mb as o_mb
from oracle import mc as o_mc
from oracle import optim as o_opt

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rel(a, b, floor=1e-3):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    return float((a - b).abs().max() / max(float(b.abs().max()), floor))


def test_mb_eval_matches_reference(gold):
    g = gold("mb.pt")
    P = gold("best_improved_model.pth")["model_state_dict"]
    for c in g["eval"]:
        x = (synth.mb_clips_bright if c["bright"] else synth.mb_clips)(c["B"], c["T"], c["H"], c["W"], c["seed"])
        with torch.no_grad():
            s, a, f = o_mb.mb_forward(P, x)
        assert rel(s, c["scores"]) < 1e-5 and rel(a, c["adj"]) < 1e-5 and rel(f, c["feat"]) < 1e-5
    assert rel(g["eval"][0]["scores"].flatten(), g["known_answers"]["scores_T8"]) < 1e-5


def test_mb_train_loss_and_grads_match_reference(gold):
    g = gold("mb.pt")
    P0 = gold("best_improved_model.pth")["model_state_dict"]
    for c in g["train"]:
        P = {k: v.clone().requires_grad_(True) for k, v in P0.items()}
        x = synth.mb_clips_bright(c["B"], c["T"], 64, 64, c["seed"])
        s, a, f = o_mb.mb_forward(P, x, True, c["keep_feat"], c["keep_graph"])
        loss, comps = o_mb.mb_loss(s, a, c["pseudo"])
        loss.backward()
        assert rel(loss, c["loss"]) < 1e-5
        for k, v in c["comps"].items():
            assert abs(comps[k] - v) <= 1e-5 * max(1.0, abs(v)), k
        for k, sm in c["grad_summary"].items():
            assert abs(float(P[k].grad.double().norm()) - sm["norm"]) <= 1e-4 * max(sm["norm"], 1e-6), k


def test_mb_loss32_and_input_grads(gold):
    c = gold("mb.pt")["loss32"]
    sc = c["scores"].clone().requires_grad_(True)
    ad = c["adj"].clone().requires_grad_(True)
    loss, comps = o_mb.mb_loss(sc, ad, c["pseudo"])
    loss.backward()
    assert rel(loss, c["loss"]) < 1e-6
    assert rel(sc.grad, c["dscores"]) < 1e-5 and rel(ad.grad, c["dadj"]) < 1e-5


def test_mb_trajectory_with_oracle_optimizer(gold):
    """3 AdamW steps from the shipped checkpoint incl. its optimizer state (s2:221-238)."""
    g = gold("mb.pt")["trajectory"]
    ck = gold("best_improved_model.pth")
    names = list(ck["model_state_dict"].keys())
    P = {k: v.clone() for k, v in ck["model_state_dict"].items()}
    st = ck["optimizer_state_dict"]["state"]
    M = {k: st[i]["exp_avg"].clone() for i, k in enumerate(names)}
    V = {k: st[i]["exp_avg_sq"].clone() for i, k in enumerate(names)}
    step = int(st[0]["step"])
    for it, sd in enumerate(g["seeds"]):
        Pg = {k: v.clone().requires_grad_(True) for k, v in P.items()}
        x = synth.mb_clips_bright(8, 8, 64, 64, sd)
        kf, kg = synth.keep_mask((8, 16), 0.3, sd + 1), synth.keep_mask((8, 128), 0.3, sd + 2)
        pseudo = (g["steps"][it]["u"] > 0.95).float()
        s, a, f = o_mb.mb_forward(Pg, x, True, kf, kg)
        loss, _ = o_mb.mb_loss(s, a, pseudo)
        loss.backward()
        assert abs(float(loss) - g["losses"][it]) < 1e-5 * max(1, abs(g["losses"][it]))
        norm, grads = o_opt.clip_grad_norm([Pg[k].grad for k in names], 0.5)
        assert abs(float(norm) - g["steps"][it]["grad_norm"]) < 1e-4 * g["steps"][it]["grad_norm"]
        step += 1
        for k, gr in zip(names, grads):
            P[k], M[k], V[k] = o_opt.adamw_step(P[k], gr, M[k], V[k], step, 5e-4, weight_decay=1e-3)
    for k, v in g["final_small"].items():
        assert rel(P[k], v) < 1e-5, k
    assert step == g["final_opt_step"]


@pytest.fixture
def golden_threads():
    """The CPU thread count tools/make_golden.py computed the fixtures with.  The conv3d backward's reduction order follows the thread
    count, and so does the round-off that forms a BatchNorm-fed bias's analytically zero gradient (M-C features.0.bias)."""
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


def test_mc_matches_reference(gold, golden_threads):
    g = gold("mc.pt")
    synth_state = synth.synth_fill(g["init_state"], seed=g["state_seed"])
    for k in synth_state:
        if k.startswith("classifier") and k.endswith("weight"):
            synth_state[k] = synth_state[k] * 3.0
    for c in g["eval"]:
        st = g["init_state"] if c["weights"] == "init" else synth_state
        x = synth.mc_clips(c["B"], c["T"], c["H"], c["W"], c["seed"])
        with torch.no_grad():
            s = o_mc.mc_forward(st, x)
        assert rel(s, c["scores"]) < 1e-5
    for c in g["train"]:
        P = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v.clone())
             for k, v in synth_state.items()}
        x = synth.mc_clips(c["B"], c["T"], 64, 64, c["seed"])
        ns = {}
        s = o_mc.mc_forward(P, x, True, c["keep0"], c["keep1"], ns)
        loss = o_mc.bce(s, c["y"])
        loss.backward()
        assert rel(loss, c["loss"]) < 1e-5
        gscale = max(float(v.abs().max()) for v in c["grads"].values())
        for k, v in c["grads"].items():
            assert rel(P[k].grad, v, floor=gscale) < 1e-4, k
        for k, v in c["new_stats"].items():
            assert rel(ns[k].float(), v.float()) < 1e-5, k


def test_ma_matches_reference(gold):
    from oracle.ma import ma_forward, ma_loss
    g = gold("ma.pt")
    import torch.nn as nn
    for c in g["cases"]:
        P = ma_synth_state(c["seed"], c["live"])
        x = synth.ma_clips(c["B"], c["T"], c["H"], c["W"], c["xseed"], c["wide"])
        eps, keep = ma_noise(c)
        with torch.no_grad():
            out = ma_forward(P, x, eps, c["train"], keep)
            loss, comps = ma_loss(out, c["labels"])
        assert rel(out["anomaly_scores"], c["anomaly_scores"]) < 1e-4
        assert rel(out["direct_predictions"], c["direct_predictions"]) < 1e-4
        assert rel(out["kl_losses"], c["kl_losses"]) < 1e-4
        assert torch.equal(out["det_counts"], c["det_counts"])
        assert rel(loss, c["loss"]) < 1e-4


# ---- shared helpers for M-A fixtures (also used by the GPU tests) -------------------------------------------------
def ma_reference_shapes():
    """state_dict skeleton of causal_anomaly_detection.CausalAnomalyDetector (cad:508-538), built without the reference."""
    import collections
    sd = collections.OrderedDict()

    def conv(name, co, ci, k):
        sd[name + ".weight"] = torch.zeros(co, ci, k, k)
        sd[name + ".bias"] = torch.zeros(co)

    def bn(name, c):
        sd[name + ".weight"] = torch.ones(c); sd[name + ".bias"] = torch.zeros(c)
        sd[name + ".running_mean"] = torch.zeros(c); sd[name + ".running_var"] = torch.ones(c)
        sd[name + ".num_batches_tracked"] = torch.tensor(0)

    def lin(name, o, i):
        sd[name + ".weight"] = torch.zeros(o, i)
        sd[name + ".bias"] = torch.zeros(o)

    conv("backbone.conv1", 32, 1, 7); bn("backbone.bn1", 32)
    cin = 32
    for li, co in zip((1, 2, 3, 4), (32, 64, 128, 256)):
        conv(f"backbone.layer{li}.0", co, cin, 3); bn(f"backbone.layer{li}.1", co)
        conv(f"backbone.layer{li}.3", co, co, 3); bn(f"backbone.layer{li}.4", co)
        cin = co
    for idx, (o, i) in zip((0, 3, 6, 8, 10), ((512, 6144), (256, 512), (128, 256), (64, 128), (20, 64))):
        lin(f"detector.detector_net.{idx}", o, i)
    for idx, (o, i) in zip((0, 2, 4), ((32, 4), (64, 32), (64, 64))):
        lin(f"tracker.reid_net.{idx}", o, i)
    sd["traj_encoder.gru.weight_ih_l0"] = torch.zeros(192, 68); sd["traj_encoder.gru.weight_hh_l0"] = torch.zeros(192, 64)
    sd["traj_encoder.gru.bias_ih_l0"] = torch.zeros(192); sd["traj_encoder.gru.bias_hh_l0"] = torch.zeros(192)
    lin("traj_encoder.encoder", 32, 64)
    lin("causal_extractor.encoder.0", 32, 32); lin("causal_extractor.encoder.2", 32, 32)
    lin("causal_extractor.mu_head", 6, 32); lin("causal_extractor.logvar_head", 6, 32)
    sd["structure_learner.structure_params"] = torch.zeros(6, 6)
    lin("structure_learner.node_encoder", 32, 6)
    lin("structure_learner.edge_predictor.0", 32, 64); lin("structure_learner.edge_predictor.2", 1, 32)
    for idx, (o, i) in zip((0, 2, 4), ((32, 6), (32, 32), (6, 32))):
        lin(f"dynamics_predictor.dynamics_net.{idx}", o, i)
    for idx, (o, i) in zip((0, 3, 5), ((64, 18), (32, 64), (1, 32))):
        lin(f"anomaly_scorer.causal_scorer.{idx}", o, i)
    for idx, (o, i) in zip((0, 2, 4), ((32, 12), (16, 32), (1, 16))):
        lin(f"anomaly_scorer.motion_scorer.{idx}", o, i)
    for idx, (o, i) in zip((0, 2, 4), ((32, 6), (16, 32), (1, 16))):
        lin(f"anomaly_scorer.temporal_scorer.{idx}", o, i)
    for idx, (o, i) in zip((0, 3, 6, 8, 10), ((512, 6144), (256, 512), (128, 256), (64, 128), (2, 64))):
        lin(f"direct_classifier.{idx}", o, i)
    return sd


DET_BIAS_SAT = [180, 120, 25, 50, 150, 100, 20, 45, 210, 140, 30, 55, 120, 80, 22, 48, 240, 160, 28, 52]     # cad:186-192
DET_BIAS_LIVE = [0.0, 0.0, -0.5, -0.5, 0.3, -0.2, 0.0, 0.2, -3.5, 0.1, 0.0, 0.0, 0.4, 3.5, 0.0, 0.0, 0.1, -0.1, 4.5, 0.0]


def ma_synth_state(seed, live):
    sd = ma_reference_shapes()
    sd["detector.detector_net.10.bias"] = torch.tensor(DET_BIAS_SAT, dtype=torch.float32)
    P = synth.synth_fill(sd, seed=seed, skip=("detector.detector_net.10.bias",))
    if live:
        P["detector.detector_net.10.bias"] = torch.tensor(DET_BIAS_LIVE)
        P["detector.detector_net.10.weight"] = P["detector.detector_net.10.weight"] * 24.0
    return P


def ma_noise(c):
    B, T, xs = c["B"], c["T"], c["xseed"]
    eps = torch.randn(B, 5, 6, generator=synth.gen(xs + 1))
    keep = {"det0": synth.keep_mask((B, T, 512), 0.3, xs + 2), "det1": synth.keep_mask((B, T, 256), 0.2, xs + 3),
            "scorer0": synth.keep_mask((B, 64), 0.2, xs + 4), "cls0": synth.keep_mask((B, 512), 0.3, xs + 5),
            "cls1": synth.keep_mask((B, 256), 0.2, xs + 6)}
    return eps, keep



# ---- M-A0 (video_anomaly_detection.py) ------------------------------------------------------------------------------
def ma0_reference_shapes():
    """state_dict skeleton of video_anomaly_detection.CausalAnomalyDetector (vad:405-417), built without the reference: cad's backbone,
    tracker, GRU encoder, factor extractor, structure learner and dynamics net around vad's two-head detector and single scorer."""
    import collections
    full = ma_reference_shapes()
    sd = collections.OrderedDict()
    for k, v in full.items():
        if k.startswith("detector."):
            if "detector.bbox_head.weight" not in sd:
                sd["detector.bbox_head.weight"] = torch.zeros(12, 6144); sd["detector.bbox_head.bias"] = torch.zeros(12)
                sd["detector.conf_head.weight"] = torch.zeros(3, 6144); sd["detector.conf_head.bias"] = torch.zeros(3)
            continue
        if k.startswith("anomaly_scorer.") or k.startswith("direct_classifier."):
            continue
        sd[k] = v
    for idx, (o, i) in zip((0, 2, 4), ((32, 18), (16, 32), (1, 16))):
        sd[f"anomaly_scorer.score_net.{idx}.weight"] = torch.zeros(o, i)
        sd[f"anomaly_scorer.score_net.{idx}.bias"] = torch.zeros(o)
    return sd


def ma0_synth_state(seed, margin):
    P = synth.synth_fill(ma0_reference_shapes(), seed=seed)
    if not margin:
        P["detector.conf_head.weight"] = P["detector.conf_head.weight"] * 4.0
    else:
        P["detector.conf_head.weight"] = P["detector.conf_head.weight"] * 0.02
        P["detector.conf_head.bias"] = torch.tensor([1.5, -1.5, 0.8])
    return P


def ma0_input(c):
    if c.get("stream"):
        seq = synth.ma_clips(1, c["T"] + 4 * (c["B"] - 1), c["H"], c["W"], c["xseed"], c["wide"])[0]
        return torch.stack([seq[4 * w: 4 * w + c["T"]] for w in range(c["B"])]), seq
    return synth.ma_clips(c["B"], c["T"], c["H"], c["W"], c["xseed"], c["wide"]), None


def ma0_eps(c):
    return torch.randn(c["B"], 5, 6, generator=synth.gen(c["xseed"] + 1))


def test_ma0_matches_reference(gold):
    """oracle/ma0.py against the unmodified video_anomaly_detection.py (tests/golden/ma0.pt): ragged detections (0..3 anchors per frame),
    scores, KL, adjacency, 2-term loss."""
    from oracle.ma0 import ma0_forward, ma0_loss
    seen = set()
    for c in gold("ma0.pt")["cases"]:
        P = ma0_synth_state(c["seed"], c["margin"])
        x, _ = ma0_input(c)
        with torch.no_grad():
            out = ma0_forward(P, x, ma0_eps(c), c["train"])
            loss, comps = ma0_loss(out, c["labels"])
        assert rel(out["anomaly_scores"], c["anomaly_scores"]) < 1e-4
        assert rel(out["kl_losses"], c["kl_losses"]) < 1e-4
        assert rel(out["adjacency_matrices"], c["adjacency"]) < 1e-4
        assert torch.equal(out["det_counts"], c["det_counts"]) and torch.equal(out["det_real"], c["det_real"])
        assert rel(loss, c["loss"]) < 1e-4
        seen |= set(c["det_real"].flatten().tolist())
    assert seen == {0, 1, 2, 3}, seen          # the fixtures cover the dummy box and every anchor count


def test_ma_c2_benchmarked_shape_forward_matches_reference(gold):
    """The oracle at the benchmarked shape (32 x 16 x 240 x 360, train-mode BatchNorm, injected dropout / eps): scores and the 4-term
    loss of the unmodified reference (tests/golden/ma_c2.pt).  Forward only here (the backward is asserted when the fixture is made)."""
    c = gold("ma_c2.pt")["cases"][0]
    P = ma_synth_state(c["seed"], c["live"])
    x = synth.ma_clips(c["B"], c["T"], c["H"], c["W"], c["xseed"], c["wide"])
    eps, keep = ma_noise(c)
    with torch.no_grad():
        out = o_ma.ma_forward(P, x, eps, True, keep, {})
        loss, comps = o_ma.ma_loss(out, c["labels"])
    assert rel(out["anomaly_scores"], c["anomaly_scores"]) < 1e-5
    assert rel(loss, c["loss"]) < 1e-5
    for k, v in c["comps"].items():
        assert abs(comps[k] - v) <= 1e-5 * max(1.0, abs(v)), k


def test_ma_trajectory_oracle_vs_reference_train_model(gold):
    """oracle.train.ma_train_step (the CPU stand-in bench.py times when the reference copy is absent) against three iterations of
    the reference's own train_model loop (cad:637-693): per-step losses and the final parameters."""
    from oracle import train as o_train
    g = gold("ma_traj.pt")["traj_live"]
    B, T = g["B"], g["T"]
    P0 = ma_synth_state(g["seed"], g["live"])
    P = {k: v.clone() for k, v in P0.items()}
    opt = o_train.OracleAdam(o_train.ma_trainable(P), 3e-4, 1e-5, True, 1.0)
    losses = []
    for xs in g["xseeds"]:
        x = synth.ma_clips(B, T, g["H"], g["W"], xs, g["wide"])
        y = (torch.rand(B, generator=synth.gen(xs + 9)) < 0.5).long()
        eps, keep = ma_noise({"B": B, "T": T, "xseed": xs})
        losses.append(o_train.ma_train_step(P, opt, x, y, eps, keep)[0])
    assert abs(sum(losses) / 3 - g["mean_loss"]) < 1e-5 * g["mean_loss"]

    def sample(t):              # the fixture keeps at most sample_cap elements of each tensor's strided sample
        return synth.strided_sample(synth.strided_sample(t), g["sample_cap"])
    for k, ref in g["final_sample"].items():
        if "running" in k or synth.is_bn_fed_conv_bias(k):
            continue
        moved = float((ref - sample(P0[k])).double().norm())
        d = float((sample(P[k]) - ref).double().norm())
        assert d <= 0.25 * moved + 1e-12, (k, d, moved)


# --------------------------------------------------------------------------------------------------------- M-D
def md_synth_state(seed):
    """The state tools/make_golden.py gave the reference VideoAutoEncoder (rebuilt from seeds, no reference needed)."""
    import torch.nn as nn
    torch.manual_seed(seed)
    keys = {}
    enc = [(1, 32), (32, 64), (64, 128), (128, 128)]
    for i, (ci, co) in enumerate(enc):
        keys[f"encoder.{3 * i}.weight"] = torch.zeros(co, ci, 4, 4)
        keys[f"encoder.{3 * i}.bias"] = torch.zeros(co)
        for n_, v in (("weight", torch.ones(co)), ("bias", torch.zeros(co)), ("running_mean", torch.zeros(co)), ("running_var", torch.ones(co)),
                      ("num_batches_tracked", torch.tensor(0))):
            keys[f"encoder.{3 * i + 1}.{n_}"] = v
    keys["encoder.13.weight"], keys["encoder.13.bias"] = torch.zeros(64, 2048), torch.zeros(64)
    keys["decoder.0.weight"], keys["decoder.0.bias"] = torch.zeros(2048, 64), torch.zeros(2048)
    dec = [(128, 128), (128, 64), (64, 32)]
    for i, (ci, co) in enumerate(dec):
        keys[f"decoder.{3 * i + 3}.weight"] = torch.zeros(ci, co, 4, 4)
        keys[f"decoder.{3 * i + 3}.bias"] = torch.zeros(co)
        for n_, v in (("weight", torch.ones(co)), ("bias", torch.zeros(co)), ("running_mean", torch.zeros(co)), ("running_var", torch.ones(co)),
                      ("num_batches_tracked", torch.tensor(0))):
            keys[f"decoder.{3 * i + 4}.{n_}"] = v
    keys["decoder.12.weight"], keys["decoder.12.bias"] = torch.zeros(32, 1, 4, 4), torch.zeros(1)
    for n_, shp in (("weight_ih_l0", (256, 64)), ("weight_hh_l0", (256, 64)), ("bias_ih_l0", (256,)), ("bias_hh_l0", (256,))):
        keys[f"temporal_encoder.{n_}"] = torch.zeros(shp)
    keys["normal_memory"] = torch.zeros(500, 64)
    keys["memory_ptr"] = torch.zeros(1, dtype=torch.long)
    keys["temperature"] = torch.tensor(1.0)
    return keys


def md_state_like(model_state, seed):
    """synth_fill in the REFERENCE's state_dict key order + the partly filled memory bank used by the golden generator."""
    sd = synth.synth_fill(model_state, 700 + seed, skip=("normal_memory", "memory_ptr", "temperature", "num_batches_tracked"))
    sd["normal_memory"] = torch.zeros(500, 64)
    sd["normal_memory"][:37] = torch.randn(37, 64, generator=synth.gen(900 + seed))
    sd["memory_ptr"] = torch.tensor([37])
    return sd


def md_reference_order(keys, order):
    """Re-order to the reference module's state_dict key order (recorded in the fixture)."""
    assert set(order) == set(keys), set(order) ^ set(keys)
    return {k: keys[k] for k in order}


def test_md_oracle_matches_reference(gold):
    from oracle import md as o_md
    g = gold("md.pt")
    for c in g["cases"]:
        P = md_state_like(md_reference_order(md_synth_state(c["seed"]), c["state_keys"]), c["seed"])
        x = synth.md_clips(c["B"], c["T"], seed=c["xseed"])
        if c["train"]:
            for k, v in P.items():
                if v.is_floating_point() and "running" not in k and k not in ("normal_memory", "temperature"):
                    v.requires_grad_(True)
        rec, z, ff, ms = o_md.md_forward(P, x, c["train"])
        assert rel(rec[:, 0], c["recon_frame0"]) < 1e-5, c["name"]
        assert rel(z, c["sequence_feature"]) < 1e-5 and rel(ff, c["frame_features"]) < 1e-5
        assert rel(ms, c["anomaly_score"], floor=1e-6) < 1e-5
        if not c["train"]:
            assert rel(o_md.combined_scores(x, rec, ms), c["combined"]) < 1e-5
        else:
            loss = o_md.recon_loss(x, rec)
            assert abs(float(loss) - c["loss"]) < 1e-6
            loss.backward()
            gmax = max(v["norm"] for v in c["grads"].values())
            for k, gs in c["grads"].items():
                assert abs(float(P[k].grad.double().norm()) - gs["norm"]) < 5e-3 * gmax, k
            o_md.update_memory(P, z)
            for k, v in c["new_stats"].items():
                assert rel(P[k].detach().float(), v.float(), floor=1e-6) < 1e-5, k
            assert rel(P["normal_memory"][37:37 + c["B"]].detach(), c["memory_rows"]) < 1e-5
