"""Generate tests/golden/*.pt by running the UNMODIFIED reference from /root/reference on CPU and
assert that the oracle restatement (oracle/) reproduces it.  Build-container only.

    python tools/make_golden.py [mb] [mc] [ma]

Each fixture stores seeds + (small) tensors; big inputs / weights are rebuilt from tests/synth.py.
"""
from __future__ import annotations

import contextlib
import copy
import io
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import synth  # noqa: E402
from oracle.ref_harness import NoiseInjector, import_ref  # noqa: E402

from oracle import ma as o_ma  # noqa: E402
from oracle import ma0 as o_ma0  # noqa: E402
from oracle import mb as o_mb  # noqa: E402
from oracle import mc as o_mc  # noqa: E402
from oracle import md as o_md  # noqa: E402
from oracle import optim as o_opt  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
# elements kept of each final parameter's strided sample in ma_traj.pt (keeps the fixture under 1 MB)
TRAJ_SAMPLE_CAP = 3072
torch.set_num_threads(8)


def close(a, b, tol, what, floor=1e-3):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    err = (a - b).abs().max().item() if a.numel() else 0.0
    ref = b.abs().max().item() if b.numel() else 0.0
    ok = err <= tol * max(ref, floor)
    print(f"   {'ok ' if ok else 'BAD'} {what}: max|d|={err:.3e} (ref max {ref:.3e})")
    assert ok, what


# --------------------------------------------------------------------------------------------- M-B
def make_mb():
    print("== M-B (avenue_training_script2.py) ==")
    s2 = import_ref("avenue_training_script2")
    ck = torch.load(os.path.join(os.path.dirname(s2.__file__), "best_improved_model.pth"), map_location="cpu", weights_only=False)
    synth.save_golden_checkpoint(ck, "best_improved_model.pth")
    P = ck["model_state_dict"]
    out = {"eval": [], "known_answers": {
        "scores_T8": [0.13723799586296082, 0.13770483434200287, 0.13747946918010712, 0.13792464137077332],
        "scores_T16": [0.12867575883865356, 0.12878333032131195, 0.1282607465982437, 0.12863218784332275]}}

    model = s2.CausalAnomalyDetector()
    model.load_state_dict(P, strict=True)
    model.eval()
    for (B, T, H, W, seed, bright) in [(4, 8, 64, 64, 1234, False), (4, 16, 64, 64, 1234, False), (3, 12, 48, 48, 7, True),
                                       (1, 8, 64, 64, 9, False), (2, 64, 64, 64, 21, True), (5, 9, 40, 56, 33, True)]:
        x = synth.mb_clips_bright(B, T, H, W, seed) if bright else synth.mb_clips(B, T, H, W, seed)
        with torch.no_grad():
            s, a, f = model(x)
            so, ao, fo = o_mb.mb_forward(P, x)
        print(f" eval B{B} T{T} {H}x{W}")
        close(so, s, 1e-6, "oracle scores"); close(ao, a, 1e-6, "oracle adj"); close(fo, f, 1e-6, "oracle feat")
        out["eval"].append({"B": B, "T": T, "H": H, "W": W, "seed": seed, "bright": bright,
                            "scores": s.clone(), "adj": a.clone(), "feat": f.clone()})
    close(out["eval"][0]["scores"].flatten(), out["known_answers"]["scores_T8"], 1e-5, "SURVEY known answers T8")
    close(out["eval"][1]["scores"].flatten(), out["known_answers"]["scores_T16"], 1e-5, "SURVEY known answers T16")

    # ---- one training forward/loss/backward with injected noise (s2:221-236)
    def train_case(B, T, seed, n_anom):
        x = synth.mb_clips_bright(B, T, 64, 64, seed)
        kf = synth.keep_mask((B, 16), 0.3, seed + 1)
        kg = synth.keep_mask((B, 128), 0.3, seed + 2)
        u = torch.rand(B, generator=synth.gen(seed + 3)) * 0.9
        u[:n_anom] = 0.99                      # rand_like(targets) > 0.95 -> pseudo label 1
        pseudo = (u > 0.95).float()
        trainer = s2.ImprovedMiniCausalVAD(device="cpu")
        trainer.model.load_state_dict(P, strict=True)
        trainer.model.train()
        with NoiseInjector() as inj:
            inj.dropout[id(trainer.model.feature_extractor.dropout)] = [kf]
            inj.dropout[id(trainer.model.graph_encoder[2])] = [kg]
            inj.rand = [u]
            trainer.optimizer.zero_grad()
            s, a, f = trainer.model(x)
            loss, comps = trainer.compute_improved_loss(s, a, torch.zeros(B), f)
            loss.backward()
        grads = {k: p.grad.clone() for k, p in trainer.model.named_parameters()}
        # oracle
        Pg = {k: v.clone().requires_grad_(True) for k, v in P.items()}
        so, ao, fo = o_mb.mb_forward(Pg, x, True, kf, kg)
        lo, co = o_mb.mb_loss(so, ao, pseudo)
        lo.backward()
        print(f" train B{B} T{T}")
        close(lo, loss, 1e-6, "oracle loss")
        for k in comps:
            close(co[k], comps[k], 1e-5, f"oracle comp {k}")
        for k in grads:
            close(Pg[k].grad, grads[k], 2e-5, f"oracle grad {k}")
        return {"B": B, "T": T, "seed": seed, "keep_feat": kf, "keep_graph": kg, "pseudo": pseudo, "u": u,
                "loss": loss.detach().clone(), "comps": comps, "scores": s.detach().clone(), "adj": a.detach().clone(),
                "feat": f.detach().clone(),
                "grads": {k: (g if g.numel() <= 8192 else None) for k, g in grads.items()},
                "grad_summary": {k: synth.summarize(g) for k, g in grads.items()}}

    out["train"] = [train_case(8, 8, 11, 1), train_case(4, 8, 12, 0), train_case(6, 16, 13, 2)]

    # ---- loss-only case at B=32 (K11 parity incl. d/dscores, d/dadj)
    g = synth.gen(77)
    sc = (torch.rand(32, 1, generator=g) * 0.5 + 0.05).requires_grad_(True)
    ad = (torch.rand(32, 16, 16, generator=g) * (1 - torch.eye(16))).requires_grad_(True)
    u = torch.rand(32, generator=g)
    u[3] = 0.97; u[17] = 0.999
    trainer = s2.ImprovedMiniCausalVAD(device="cpu")
    with NoiseInjector() as inj:
        inj.rand = [u]
        loss, comps = trainer.compute_improved_loss(sc, ad, torch.zeros(32), None)
        loss.backward()
    lo, co = o_mb.mb_loss(sc.detach(), ad.detach(), (u > 0.95).float())
    close(lo, loss, 1e-6, "oracle loss B32")
    out["loss32"] = {"scores": sc.detach().clone(), "adj": ad.detach().clone(), "u": u, "pseudo": (u > 0.95).float(),
                     "loss": loss.detach().clone(), "comps": comps, "dscores": sc.grad.clone(), "dadj": ad.grad.clone()}

    # ---- 3-step trajectory from the shipped checkpoint incl. AdamW state (s2:221-238)
    trainer = s2.ImprovedMiniCausalVAD(device="cpu")
    trainer.model.load_state_dict(P, strict=True)
    trainer.optimizer.load_state_dict(copy.deepcopy(ck["optimizer_state_dict"]))
    trainer.model.train()
    traj = {"B": 8, "T": 8, "seeds": [101, 102, 103], "losses": [], "steps": []}
    for sd in traj["seeds"]:
        x = synth.mb_clips_bright(8, 8, 64, 64, sd)
        kf = synth.keep_mask((8, 16), 0.3, sd + 1); kg = synth.keep_mask((8, 128), 0.3, sd + 2)
        u = torch.rand(8, generator=synth.gen(sd + 3))
        with NoiseInjector() as inj:
            inj.dropout[id(trainer.model.feature_extractor.dropout)] = [kf]
            inj.dropout[id(trainer.model.graph_encoder[2])] = [kg]
            inj.rand = [u]
            trainer.optimizer.zero_grad()
            s, a, f = trainer.model(x)
            loss, comps = trainer.compute_improved_loss(s, a, torch.zeros(8), f)
            loss.backward()
            norm = torch.nn.utils.clip_grad_norm_(trainer.model.parameters(), max_norm=0.5)
            trainer.optimizer.step()
        traj["losses"].append(float(loss)); traj["steps"].append({"comps": comps, "grad_norm": float(norm), "u": u})
    traj["final_summary"] = {k: synth.summarize(v) for k, v in trainer.model.state_dict().items()}
    traj["final_small"] = {k: v.clone() for k, v in trainer.model.state_dict().items() if v.numel() <= 8192}
    traj["final_opt_step"] = float(trainer.optimizer.state_dict()["state"][0]["step"])
    out["trajectory"] = traj
    print(" trajectory losses", traj["losses"])
    torch.save(out, os.path.join(GOLD, "mb.pt"))


# --------------------------------------------------------------------------------------------- M-C
def make_mc():
    print("== M-C (minicausal_vad_complete3.py) ==")
    mc3 = import_ref("minicausal_vad_complete3")
    torch.manual_seed(0)
    model = mc3.SimpleVideoAnomalyDetector()
    out = {"init_state": {k: v.clone() for k, v in model.state_dict().items()}, "eval": [], "train": []}
    # "trained-like" weights: reproducible, non-degenerate (the stock init gives a constant 0.5)
    P = synth.synth_fill(model.state_dict(), seed=5)
    for k in P:
        if k.startswith("classifier") and k.endswith("weight"):
            P[k] = P[k] * 3.0
    out["state_seed"] = 5
    model.load_state_dict(P, strict=True)
    for name, st in (("init", out["init_state"]), ("synth", P)):
        model.load_state_dict(st, strict=True)
        model.eval()
        for (B, T, H, W, seed) in [(4, 16, 64, 64, 1234), (2, 64, 64, 64, 3), (2, 10, 36, 44, 8), (1, 4, 64, 64, 2)]:
            x = synth.mc_clips(B, T, H, W, seed)
            with torch.no_grad():
                s = model(x)
                so = o_mc.mc_forward(st, x)
            print(f" eval[{name}] B{B} T{T} {H}x{W}  scores {s.flatten()[:3].tolist()}")
            close(so, s, 1e-6, "oracle scores")
            out["eval"].append({"weights": name, "B": B, "T": T, "H": H, "W": W, "seed": seed, "scores": s.clone()})
    # training step: forward (batch-stat BN) + BCE + backward
    for (B, T, seed) in [(4, 8, 41), (6, 16, 42)]:
        model.load_state_dict(P, strict=True)
        model.train()
        x = synth.mc_clips(B, T, 64, 64, seed)
        y = (torch.rand(B, generator=synth.gen(seed + 5)) > 0.5).float()
        k0 = synth.keep_mask((B, 32), 0.5, seed + 1); k1 = synth.keep_mask((B, 16), 0.3, seed + 2)
        with NoiseInjector() as inj:
            inj.dropout[id(model.classifier[0])] = [k0]
            inj.dropout[id(model.classifier[3])] = [k1]
            model.zero_grad()
            s = model(x)
            loss = torch.nn.BCELoss()(s.squeeze(), y)
            loss.backward()
        grads = {k: p.grad.clone() for k, p in model.named_parameters()}
        new_state = {k: v.clone() for k, v in model.state_dict().items() if "running" in k or "num_batches" in k}
        Pg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v.clone()) for k, v in P.items()}
        ns = {}
        so = o_mc.mc_forward(Pg, x, True, k0, k1, ns)
        lo = o_mc.bce(so, y)
        lo.backward()
        print(f" train B{B} T{T} loss {float(loss):.6f}")
        close(lo, loss, 1e-6, "oracle loss")
        gscale = max(float(g.abs().max()) for g in grads.values())
        for k in grads:
            close(Pg[k].grad, grads[k], 5e-5, f"oracle grad {k}", floor=gscale)
        for k in new_state:
            close(ns[k], new_state[k], 1e-5, f"oracle stat {k}")
        out["train"].append({"B": B, "T": T, "seed": seed, "y": y, "keep0": k0, "keep1": k1, "loss": loss.detach().clone(),
                             "scores": s.detach().clone(), "grads": grads, "new_stats": new_state})
    # 3-step Adam trajectory following mc3:269-311 (clip only when norm > 10)
    model.load_state_dict(P, strict=True)
    model.train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=1e-5, eps=1e-8)
    traj = {"B": 4, "T": 8, "seeds": [51, 52, 53], "losses": []}
    for sd in traj["seeds"]:
        x = synth.mc_clips(4, 8, 64, 64, sd)
        y = (torch.rand(4, generator=synth.gen(sd + 5)) > 0.5).float()
        k0 = synth.keep_mask((4, 32), 0.5, sd + 1); k1 = synth.keep_mask((4, 16), 0.3, sd + 2)
        with NoiseInjector() as inj:
            inj.dropout[id(model.classifier[0])] = [k0]
            inj.dropout[id(model.classifier[3])] = [k1]
            opt.zero_grad()
            s = model(x).squeeze()
            loss = torch.nn.BCELoss()(s, y)
            loss.backward()
            gn = sum(p.grad.data.norm(2).item() ** 2 for p in model.parameters()) ** 0.5
            if gn > 10.0:
                torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
            opt.step()
        traj["losses"].append(float(loss))
    traj["final"] = {k: v.clone() for k, v in model.state_dict().items()}
    out["trajectory"] = traj
    print(" trajectory losses", traj["losses"])
    torch.save(out, os.path.join(GOLD, "mc.pt"))


# --------------------------------------------------------------------------------------------- M-A
def ma_state(cad, seed, live_detector):
    torch.manual_seed(0)
    model = cad.CausalAnomalyDetector()
    P = synth.synth_fill(model.state_dict(), seed=seed, skip=("detector.detector_net.10.bias",))
    if live_detector:
        # un-saturate the detector so 0..5 boxes per frame pass the validity window (cad:217-218)
        P["detector.detector_net.10.bias"] = torch.tensor(
            [0.0, 0.0, -0.5, -0.5, 0.3, -0.2, 0.0, 0.2, -3.5, 0.1, 0.0, 0.0, 0.4, 3.5, 0.0, 0.0, 0.1, -0.1, 4.5, 0.0])
        P["detector.detector_net.10.weight"] = P["detector.detector_net.10.weight"] * 24.0
    return model, P


def ref_ma_run(cad, model, P, x, labels, eps, ntr, train, keep):
    """Run the reference model + its 4-term loss (cad:671-688, the non-AMP branch) with injected noise."""
    model.load_state_dict(P, strict=True)
    cad.apply_memory_efficient_training.__globals__["print"] = lambda *a, **k: None
    cad.apply_memory_efficient_training(model)
    model.train(train)
    B = x.shape[0]
    with NoiseInjector() as inj:
        inj.randn = [eps[b, : int(ntr[b])].clone() for b in range(B)]
        if train:
            inj.dropout[id(model.detector.detector_net[2])] = [keep["det0"]]
            inj.dropout[id(model.detector.detector_net[5])] = [keep["det1"]]
            inj.dropout[id(model.anomaly_scorer.causal_scorer[2])] = [keep["scorer0"][b:b + 1] for b in range(B)]
            inj.dropout[id(model.direct_classifier[2])] = [keep["cls0"]]
            inj.dropout[id(model.direct_classifier[5])] = [keep["cls1"]]
        model.zero_grad()
        ctx = torch.enable_grad() if train else torch.no_grad()
        with ctx:
            outputs = model(x)
            ce = torch.nn.CrossEntropyLoss()(outputs["direct_predictions"], labels)
            an = torch.nn.MSELoss()(outputs["anomaly_scores"], labels.float())
            kls = outputs["kl_losses"]
            kl = sum(k for k in kls if torch.isfinite(k)) / len(kls)
            cs = torch.nn.MSELoss()(outputs["causal_anomaly_scores"], labels.float())
            total = 0.4 * ce + 0.3 * an + 0.2 * cs + 0.1 * kl
        if train:
            total.backward()
    return outputs, total, {"classification": float(ce), "anomaly": float(an), "causal": float(cs), "kl": float(kl)}


def make_ma():
    print("== M-A (causal_anomaly_detection.py) ==")
    cad = import_ref("causal_anomaly_detection")
    out = {"cases": []}
    cases = [
        dict(name="sat_eval", seed=3, live=False, B=2, T=4, H=240, W=360, wide=True, train=False, xseed=1234),
        dict(name="sat_train", seed=3, live=False, B=2, T=4, H=240, W=360, wide=True, train=True, xseed=1235),
        dict(name="live_eval", seed=4, live=True, B=3, T=3, H=120, W=180, wide=False, train=False, xseed=77),
        dict(name="live_train", seed=4, live=True, B=3, T=3, H=120, W=180, wide=False, train=True, xseed=78),
    ]
    for c in cases:
        model, P = ma_state(cad, c["seed"], c["live"])
        B, T = c["B"], c["T"]
        x = synth.ma_clips(B, T, c["H"], c["W"], c["xseed"], c["wide"])
        labels = (torch.rand(B, generator=synth.gen(c["xseed"] + 9)) < 0.5).long()
        eps = torch.randn(B, 5, 6, generator=synth.gen(c["xseed"] + 1))
        keep = {"det0": synth.keep_mask((B, T, 512), 0.3, c["xseed"] + 2), "det1": synth.keep_mask((B, T, 256), 0.2, c["xseed"] + 3),
                "scorer0": synth.keep_mask((B, 64), 0.2, c["xseed"] + 4), "cls0": synth.keep_mask((B, 512), 0.3, c["xseed"] + 5),
                "cls1": synth.keep_mask((B, 256), 0.2, c["xseed"] + 6)}
        # oracle first (gives the per-clip track counts needed to size the injected eps)
        Pg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v.clone()) for k, v in P.items()}
        ns = {}
        oo = o_ma.ma_forward(Pg, x, eps, c["train"], keep, ns)
        lo, co = o_ma.ma_loss(oo, labels)
        if c["train"]:
            lo.backward()
        ro, rl, rc = ref_ma_run(cad, model, P, x, labels, eps, oo["n_tracks"], c["train"], keep)
        print(f" case {c['name']}: tracks/clip {oo['n_tracks'].tolist()} det counts {oo['det_counts'].flatten().tolist()}")
        close(oo["anomaly_scores"], ro["anomaly_scores"], 1e-5, "anomaly_scores")
        close(oo["causal_anomaly_scores"], ro["causal_anomaly_scores"], 1e-5, "causal_anomaly_scores")
        close(oo["direct_predictions"], ro["direct_predictions"], 1e-5, "direct_predictions")
        close(oo["kl_losses"], torch.stack(ro["kl_losses"]), 1e-5, "kl_losses")
        close(oo["adjacency_matrices"], torch.stack(ro["adjacency_matrices"]), 1e-5, "adjacency")
        for b in range(B):
            n = int(oo["n_tracks"][b])
            assert ro["causal_factors"][b].shape[0] == n
            close(oo["causal_factors"][b, :n], ro["causal_factors"][b], 1e-5, f"causal_factors[{b}]")
            for t in range(T):
                m = int(oo["det_counts"][b, t])
                assert ro["detections"][b][t].shape[0] == m, (ro["detections"][b][t].shape, m)
                close(oo["detections"][b, t, :m], ro["detections"][b][t], 1e-5, f"detections[{b}][{t}]") if (b + t) == 0 else None
        close(lo, rl, 1e-5, "total loss")
        rec = {**c, "labels": labels, "loss": rl.detach().clone(), "comps": rc,
               "anomaly_scores": ro["anomaly_scores"].detach().clone(),
               "causal_anomaly_scores": ro["causal_anomaly_scores"].detach().clone(),
               "direct_predictions": ro["direct_predictions"].detach().clone(),
               "kl_losses": torch.stack(ro["kl_losses"]).detach().clone(),
               "adjacency": torch.stack(ro["adjacency_matrices"]).detach().clone(),
               "causal_factors": oo["causal_factors"].detach().clone(), "n_tracks": oo["n_tracks"].clone(),
               "detections": oo["detections"].detach().clone(), "det_counts": oo["det_counts"].clone(),
               "features_summary": synth.summarize(oo["features"])}
        if c["train"]:
            gs, has = {}, {}
            gnorm = max(float(p.grad.norm()) for p in model.parameters() if p.grad is not None)
            for k, p in model.named_parameters():
                has[k] = p.grad is not None
                if p.grad is not None:
                    og = Pg[k].grad
                    if float(p.grad.norm()) > 1e-5 * gnorm:   # conv biases feeding BN: analytically zero, roundoff only
                        rel = float((og - p.grad).double().norm() / p.grad.double().norm())
                        print(f"   {'ok ' if rel < 5e-3 else 'BAD'} grad {k}: rel-L2 {rel:.2e} |g| {float(p.grad.norm()):.3e}")
                        assert rel < 5e-3, k
                    gs[k] = synth.summarize(p.grad)
                    if p.grad.numel() <= 4096:
                        gs[k]["full"] = p.grad.clone()
                elif "backbone.conv1" in k or "backbone.bn1" in k:
                    pass                       # frozen by apply_memory_efficient_training (cad:596-598)
                else:
                    og = Pg[k].grad
                    assert og is None or float(og.abs().max()) == 0.0, f"oracle grad for {k} should be none/zero"
            rec["grad_summary"] = gs
            rec["has_grad"] = has
            rec["new_stats"] = {k: v.clone() for k, v in model.state_dict().items() if "running" in k or "num_batches" in k}
            for k, v in rec["new_stats"].items():
                close(ns[k], v, 1e-5, f"stat {k}") if "conv" not in k else None
        out["cases"].append(rec)
    torch.save(out, os.path.join(GOLD, "ma.pt"))



# --------------------------------------------------------------------------------------------- M-A0
def ma0_state(vad, seed, margin):
    torch.manual_seed(0)
    model = vad.CausalAnomalyDetector()
    P = synth.synth_fill(model.state_dict(), seed=seed)
    if not margin:
        P["detector.conf_head.weight"] = P["detector.conf_head.weight"] * 4.0      # spread the confidences: 0..3 anchors pass per frame
    if margin:
        # confidences far from the 0.5 threshold and from each other: anchors 0 and 2 pass (0 first), anchor 1 never does -- the
        # detection pattern then survives bf16 round-off in the features (the ragged cases keep the natural near-0.5 confidences)
        P["detector.conf_head.weight"] = P["detector.conf_head.weight"] * 0.02
        P["detector.conf_head.bias"] = torch.tensor([1.5, -1.5, 0.8])
    return model, P


def ref_ma0_run(vad, model, P, x, labels, eps, ntr, train):
    """Run the reference model + its loss (vad:516-531, the standard-precision branch) with injected eps."""
    model.load_state_dict(P, strict=True)
    vad.apply_memory_efficient_training.__globals__["print"] = lambda *a, **k: None
    vad.apply_memory_efficient_training(model)
    model.train(train)
    B = x.shape[0]
    with NoiseInjector() as inj:
        inj.randn = [eps[b, : int(ntr[b])].clone() for b in range(B)]
        model.zero_grad()
        with (torch.enable_grad() if train else torch.no_grad()):
            outputs = model(x)
            an = torch.nn.functional.mse_loss(outputs["anomaly_scores"], labels.float())
            valid = [k for k in outputs["kl_losses"] if torch.isfinite(k)]
            kl = sum(valid) / len(valid) if valid else torch.tensor(0.0)
            total = an + 0.001 * kl
        if train:
            total.backward()
    return outputs, total, {"anomaly": float(an), "kl": float(kl)}


def make_ma0():
    print("== M-A0 (video_anomaly_detection.py) ==")
    vad = import_ref("video_anomaly_detection")
    out = {"cases": []}
    cases = [
        dict(name="rag_eval", seed=11, margin=False, B=3, T=4, H=120, W=180, wide=False, train=False, xseed=311),
        dict(name="rag_train", seed=11, margin=False, B=3, T=4, H=120, W=180, wide=False, train=True, xseed=312),
        dict(name="margin_eval", seed=12, margin=True, B=2, T=4, H=240, W=360, wide=True, train=False, xseed=313),
        dict(name="margin_train", seed=12, margin=True, B=2, T=4, H=240, W=360, wide=True, train=True, xseed=314),
        dict(name="stream", seed=12, margin=True, B=4, T=16, H=120, W=180, wide=False, train=False, xseed=315, stream=True),
    ]
    for c in cases:
        model, P = ma0_state(vad, c["seed"], c["margin"])
        B, T = c["B"], c["T"]
        if c.get("stream"):
            # B overlapping windows (stride 4) of ONE frame sequence: what ma0.StreamingWindowScorer must reproduce clip by clip
            seq = synth.ma_clips(1, T + 4 * (B - 1), c["H"], c["W"], c["xseed"], c["wide"])[0]
            x = torch.stack([seq[4 * w: 4 * w + T] for w in range(B)])
        else:
            x = synth.ma_clips(B, T, c["H"], c["W"], c["xseed"], c["wide"])
        labels = (torch.rand(B, generator=synth.gen(c["xseed"] + 9)) < 0.5).long()
        eps = torch.randn(B, 5, 6, generator=synth.gen(c["xseed"] + 1))
        Pg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v.clone()) for k, v in P.items()}
        ns = {}
        oo = o_ma0.ma0_forward(Pg, x, eps, c["train"], ns)
        lo, co = o_ma0.ma0_loss(oo, labels)
        if c["train"]:
            lo.backward()
        ro, rl, rc = ref_ma0_run(vad, model, P, x, labels, eps, oo["n_tracks"], c["train"])
        print(f" case {c['name']}: tracks/clip {oo['n_tracks'].tolist()} real detections {oo['det_real'].flatten().tolist()}")
        close(oo["anomaly_scores"], ro["anomaly_scores"], 1e-5, "anomaly_scores")
        close(oo["kl_losses"], torch.stack(ro["kl_losses"]), 1e-5, "kl_losses")
        close(oo["adjacency_matrices"], torch.stack(ro["adjacency_matrices"]), 1e-5, "adjacency")
        for b in range(B):
            n = int(oo["n_tracks"][b])
            assert ro["causal_factors"][b].shape[0] == n
            close(oo["causal_factors"][b, :n], ro["causal_factors"][b], 1e-5, f"causal_factors[{b}]")
            for t in range(T):
                m = int(oo["det_counts"][b, t])
                assert ro["detections"][b][t].shape[0] == m, (ro["detections"][b][t].shape, m)
                assert float((oo["detections"][b, t, :m] - ro["detections"][b][t]).abs().max()) <= 1e-5 * max(1.0, float(ro["detections"][b][t].abs().max()))
        close(lo, rl, 1e-5, "total loss")
        rec = {**c, "labels": labels, "loss": rl.detach().clone(), "comps": rc, "anomaly_scores": ro["anomaly_scores"].detach().clone(),
               "kl_losses": torch.stack(ro["kl_losses"]).detach().clone(), "adjacency": torch.stack(ro["adjacency_matrices"]).detach().clone(),
               "causal_factors": oo["causal_factors"].detach().clone(), "n_tracks": oo["n_tracks"].clone(),
               "detections": oo["detections"].detach().clone(), "det_counts": oo["det_counts"].clone(), "det_real": oo["det_real"].clone(),
               "features_summary": synth.summarize(oo["features"])}
        if c["train"]:
            gs, has = {}, {}
            gnorm = max(float(p.grad.norm()) for p in model.parameters() if p.grad is not None)
            for k, p in model.named_parameters():
                has[k] = p.grad is not None
                if p.grad is not None:
                    og = Pg[k].grad
                    if float(p.grad.norm()) > 1e-5 * gnorm:
                        rel = float((og - p.grad).double().norm() / p.grad.double().norm())
                        print(f"   {'ok ' if rel < 5e-3 else 'BAD'} grad {k}: rel-L2 {rel:.2e} |g| {float(p.grad.norm()):.3e}")
                        assert rel < 5e-3, k
                    gs[k] = synth.summarize(p.grad)
                    if p.grad.numel() <= 4096:
                        gs[k]["full"] = p.grad.clone()
                elif "backbone.conv1" in k or "backbone.bn1" in k:
                    pass
                else:
                    og = Pg[k].grad
                    assert og is None or float(og.abs().max()) == 0.0, f"oracle grad for {k} should be none/zero"
            rec["grad_summary"] = gs
            rec["has_grad"] = has
            rec["new_stats"] = {k: v.clone() for k, v in model.state_dict().items() if "running" in k or "num_batches" in k}
            for k, v in rec["new_stats"].items():
                close(ns[k], v, 1e-5, f"stat {k}") if "conv" not in k else None
        out["cases"].append(rec)
    torch.save(out, os.path.join(GOLD, "ma0.pt"))
    print("   wrote ma0.pt", os.path.getsize(os.path.join(GOLD, "ma0.pt")) // 1024, "KiB")


def _ma_noise_for(B, T, xseed):
    eps = torch.randn(B, 5, 6, generator=synth.gen(xseed + 1))
    keep = {"det0": synth.keep_mask((B, T, 512), 0.3, xseed + 2), "det1": synth.keep_mask((B, T, 256), 0.2, xseed + 3),
            "scorer0": synth.keep_mask((B, 64), 0.2, xseed + 4), "cls0": synth.keep_mask((B, 512), 0.3, xseed + 5),
            "cls1": synth.keep_mask((B, 256), 0.2, xseed + 6)}
    return eps, keep


def make_ma_c2():
    """M-A at the BENCHMARKED shape (BASELINE.json configs[1]: 32 clips x 16 frames x 240x360 = 512 frames per step): one training
    forward / 4-term loss / backward of the unmodified reference (cad:671-688), saturated detector (the stock init, SURVEY fact 6) and a
    live-detector variant.  The inputs are the ones bench.py uses on rank 0 (synth.ma_clips(32,16,240,360,1234,wide) and
    bernoulli(0.3) labels from seed 1243), so bench.py can check its own first step against this fixture."""
    print("== M-A at the benchmarked shape (32 x 16 x 240 x 360) ==")
    cad = import_ref("causal_anomaly_detection")
    out = {"cases": []}
    for c in (dict(name="c2_sat_train", seed=3, live=False, B=32, T=16, H=240, W=360, wide=True, train=True, xseed=1234, label_p=0.3),
              dict(name="c2_live_train", seed=4, live=True, B=32, T=16, H=240, W=360, wide=False, train=True, xseed=2234, label_p=0.5)):
        model, P = ma_state(cad, c["seed"], c["live"])
        B, T = c["B"], c["T"]
        x = synth.ma_clips(B, T, c["H"], c["W"], c["xseed"], c["wide"])
        labels = (torch.rand(B, generator=synth.gen(c["xseed"] + 9)) < c["label_p"]).long()
        eps, keep = _ma_noise_for(B, T, c["xseed"])
        Pg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v.clone()) for k, v in P.items()}
        ns = {}
        oo = o_ma.ma_forward(Pg, x, eps, True, keep, ns)
        lo, co = o_ma.ma_loss(oo, labels)
        lo.backward()
        ograd = {k: (v.grad.clone() if torch.is_tensor(v) and v.grad is not None else None) for k, v in Pg.items()}
        ntr = oo["n_tracks"].clone()
        oo = {k: (v.detach().clone() if torch.is_tensor(v) else v) for k, v in oo.items()}
        del Pg
        ro, rl, rc = ref_ma_run(cad, model, P, x, labels, eps, ntr, True, keep)
        print(f" case {c['name']}: loss {float(rl):.6f} tracks/clip {ntr.tolist()}")
        close(oo["anomaly_scores"], ro["anomaly_scores"], 1e-5, "anomaly_scores")
        close(oo["causal_anomaly_scores"], ro["causal_anomaly_scores"], 1e-5, "causal_anomaly_scores")
        close(oo["direct_predictions"], ro["direct_predictions"], 1e-5, "direct_predictions")
        close(oo["kl_losses"], torch.stack(ro["kl_losses"]), 1e-5, "kl_losses")
        close(oo["adjacency_matrices"], torch.stack(ro["adjacency_matrices"]), 1e-5, "adjacency")
        close(lo, rl, 1e-5, "total loss")
        rec = {**c, "labels": labels, "loss": rl.detach().clone(), "comps": rc,
               "anomaly_scores": ro["anomaly_scores"].detach().clone(),
               "causal_anomaly_scores": ro["causal_anomaly_scores"].detach().clone(),
               "direct_predictions": ro["direct_predictions"].detach().clone(),
               "kl_losses": torch.stack(ro["kl_losses"]).detach().clone(),
               "adjacency": torch.stack(ro["adjacency_matrices"]).detach().clone(),
               "causal_factors": oo["causal_factors"], "n_tracks": ntr, "det_counts": oo["det_counts"].clone(),
               "features_summary": synth.summarize(oo["features"])}
        gs, has = {}, {}
        gnorm = max(float(p.grad.norm()) for p in model.parameters() if p.grad is not None)
        for k, p in model.named_parameters():
            has[k] = p.grad is not None
            if p.grad is not None:
                og = ograd[k]
                if float(p.grad.norm()) > 1e-5 * gnorm:
                    r = float((og - p.grad).double().norm() / p.grad.double().norm())
                    print(f"   {'ok ' if r < 5e-3 else 'BAD'} grad {k}: rel-L2 {r:.2e} |g| {float(p.grad.norm()):.3e}")
                    assert r < 5e-3, k
                gs[k] = synth.summarize(p.grad)
                if p.grad.numel() <= 4096:
                    gs[k]["full"] = p.grad.clone()
        rec["grad_summary"], rec["has_grad"] = gs, has
        rec["new_stats"] = {k: v.clone() for k, v in model.state_dict().items() if "running" in k or "num_batches" in k}
        for k, v in rec["new_stats"].items():
            close(ns[k], v, 1e-5, f"stat {k}") if "conv" not in k else None
        out["cases"].append(rec)
        del ro, oo, ograd

    torch.save(out, os.path.join(GOLD, "ma_c2.pt"))
    print("   wrote ma_c2.pt", os.path.getsize(os.path.join(GOLD, "ma_c2.pt")) // 1024, "KiB")



def make_ma_traj():
    """3-step M-A trajectories through the reference's OWN train_model loop (cad:609-709)."""
    print("== M-A 3-step trajectories through cad.train_model ==")
    cad = import_ref("causal_anomaly_detection")
    out = {}
    # ---- 3-step trajectory through the reference's OWN train_model loop (cad:609-709, fp32 branch on CPU: AdamW lr 3e-4 wd 1e-5,
    # clip_grad_norm_ 1.0, frozen stem), and the oracle's ma_train_step (what bench.py --impl reference falls back to) against it
    from oracle import train as o_train
    for name, live, seed, (B, T, H, W), wide in (("traj_sat", False, 3, (8, 8, 240, 360), True), ("traj_live", True, 4, (6, 5, 120, 180), False)):
        model, P0 = ma_state(cad, seed, live)
        model.load_state_dict(P0, strict=True)
        xseeds = [3100 + 10 * i + (500 if live else 0) for i in range(3)]
        batches, noises = [], []
        for xs in xseeds:
            x = synth.ma_clips(B, T, H, W, xs, wide)
            y = (torch.rand(B, generator=synth.gen(xs + 9)) < 0.5).long()
            batches.append((x, y))
            noises.append(_ma_noise_for(B, T, xs))
        # the oracle first: it yields the per-clip track counts that size the injected eps of each step
        P = {k: v.clone() for k, v in P0.items()}
        opt = o_train.OracleAdam(o_train.ma_trainable(P), 3e-4, 1e-5, True, 1.0)
        o_losses, ntrs = [], []
        for (x, y), (eps, keep) in zip(batches, noises):
            with torch.no_grad():
                ntrs.append(o_ma.ma_forward(P, x, eps, True, keep, {})["n_tracks"].clone())
            l, _ = o_train.ma_train_step(P, opt, x, y, eps, keep)
            o_losses.append(l)
        cad.device = torch.device("cpu")
        with NoiseInjector() as inj:
            for (eps, keep), ntr in zip(noises, ntrs):
                inj.randn += [eps[b, : int(ntr[b])].clone() for b in range(B)]
                inj.dropout.setdefault(id(model.detector.detector_net[2]), []).append(keep["det0"])
                inj.dropout.setdefault(id(model.detector.detector_net[5]), []).append(keep["det1"])
                inj.dropout.setdefault(id(model.anomaly_scorer.causal_scorer[2]), []).extend(keep["scorer0"][b:b + 1] for b in range(B))
                inj.dropout.setdefault(id(model.direct_classifier[2]), []).append(keep["cls0"])
                inj.dropout.setdefault(id(model.direct_classifier[5]), []).append(keep["cls1"])
            buf = io.StringIO()
            with contextlib.redirect_stdout(buf):
                model, tl, vl = cad.train_model(model, batches, [], num_epochs=1, lr=3e-4)
            assert not inj.randn, "the reference consumed a different number of eps draws than the oracle predicted"
        print(f" {name}: reference mean train loss {tl[0]:.6f}; oracle per-step losses {o_losses}")
        close(sum(o_losses) / 3, tl[0], 1e-5, f"{name} mean loss over 3 steps (oracle ma_train_step vs reference train_model)")
        final = model.state_dict()
        pmax = 0.0
        for k, v in final.items():
            if v.is_floating_point():
                # Adam's first steps move every weight by ~lr whatever the size of its gradient, and an element whose gradient is
                # round-off-sized flips direction with the summation order: compare the L2 distance with the L2 distance moved
                d = float((P[k] - v).double().norm())
                moved = float((v - P0[k]).double().norm())
                if synth.is_bn_fed_conv_bias(k):
                    # a convolution bias that feeds a BatchNorm has an analytically zero gradient; the reference's autograd leaves
                    # round-off there and Adam turns round-off into +-lr steps of random sign: nothing to compare (DESIGN.md 2)
                    continue
                if moved > 0:
                    r = d / moved
                    pmax = max(pmax, r)
                else:
                    assert d == 0.0, k
        print(f"   final parameters: oracle vs reference, worst L2 distance / L2 distance moved = {pmax:.2e}")
        assert pmax < 0.25
        out[name] = {"B": B, "T": T, "H": H, "W": W, "wide": wide, "seed": seed, "live": live, "xseeds": xseeds, "mean_loss": tl[0],
                     "oracle_losses": o_losses, "n_tracks": [n.clone() for n in ntrs],
                     "final_summary": {k: synth.summarize(v) for k, v in final.items()},
                     "moved_l2": {k: float((v - P0[k]).double().norm()) for k, v in final.items() if v.is_floating_point()},
                     "sample_cap": TRAJ_SAMPLE_CAP,
                     "final_sample": {k: synth.strided_sample(synth.strided_sample(v), TRAJ_SAMPLE_CAP)
                                      for k, v in final.items() if v.is_floating_point()}}
    torch.save(out, os.path.join(GOLD, "ma_traj.pt"))
    print("   wrote ma_traj.pt", os.path.getsize(os.path.join(GOLD, "ma_traj.pt")) // 1024, "KiB")


def md_state(cad1, seed):
    """Reference VideoAutoEncoder with reproducible, trained-like weights and a partly filled memory bank."""
    torch.manual_seed(seed)
    m = cad1.VideoAutoEncoder()
    sd = synth.synth_fill(m.state_dict(), 700 + seed, skip=("normal_memory", "memory_ptr", "temperature", "num_batches_tracked"))
    sd["normal_memory"] = torch.zeros(500, 64)
    sd["normal_memory"][:37] = torch.randn(37, 64, generator=synth.gen(900 + seed))
    sd["memory_ptr"] = torch.tensor([37])
    m.load_state_dict(sd, strict=True)
    return m


def make_md():
    """M-D: eval forward + combined score, and one training step (loss, every gradient, running statistics, memory update)."""
    print("== M-D (causal_anomaly_detection1.py)")
    cad1 = import_ref("causal_anomaly_detection1")
    cases = []
    for name, B, T, train, seed in (("eval_b3_t4", 3, 4, False, 1), ("eval_b2_t8", 2, 8, False, 2), ("train_b4_t4", 4, 4, True, 3),
                                    ("train_b6_t3", 6, 3, True, 4)):
        m = md_state(cad1, seed).to("cpu")
        P0 = {k: v.clone() for k, v in m.state_dict().items()}
        x = synth.md_clips(B, T, seed=40 + seed)
        m.train(train)
        with contextlib.redirect_stdout(io.StringIO()):
            out = m(x)
        P = {k: v.clone() for k, v in P0.items()}
        rec, z, ff, ms = o_md.md_forward(P, x, train)
        close(rec, out["reconstructed"], 2e-6, f"{name} oracle reconstructed")
        close(z, out["sequence_feature"], 2e-6, f"{name} oracle sequence_feature")
        close(ff, out["frame_features"], 2e-6, f"{name} oracle frame_features")
        close(ms, out["anomaly_score"], 2e-6, f"{name} oracle anomaly_score", floor=1e-6)
        c = {"name": name, "B": B, "T": T, "train": train, "seed": seed, "xseed": 40 + seed, "state_keys": list(P0.keys()),
             "recon_frame0": out["reconstructed"][:, 0].detach().clone(), "sequence_feature": out["sequence_feature"].detach().clone(),
             "frame_features": out["frame_features"].detach().clone(), "anomaly_score": out["anomaly_score"].detach().clone()}
        if not train:
            ref_err = torch.nn.functional.mse_loss(out["reconstructed"], x, reduction="none").view(B, -1).mean(dim=1)
            comb = 0.7 * ref_err + 0.3 * out["anomaly_score"]
            close(o_md.combined_scores(x, rec, ms), comb, 2e-6, f"{name} oracle combined score")
            c["combined"] = comb.detach().clone()
        else:
            with contextlib.redirect_stdout(io.StringIO()):
                loss = cad1.reconstruction_loss(x, out["reconstructed"])
            m.update_memory(out["sequence_feature"])
            loss.backward()
            Pg = {k: v.clone().requires_grad_(v.is_floating_point() and "running" not in k and k not in ("normal_memory", "temperature"))
                  for k, v in P0.items()}
            rec2, z2, _, _ = o_md.md_forward(Pg, x, True)
            lo = o_md.recon_loss(x, rec2)
            lo.backward()
            close(lo, loss, 2e-6, f"{name} oracle loss")
            grads = {}
            gmax = max(float(p_.grad.abs().max()) for p_ in m.parameters())     # biases feeding a BatchNorm carry pure round-off
            for k, p_ in m.named_parameters():
                # per-time-step BatchNorm over B x 4 x 4 = 32..64 values amplifies fp32 round-off: two orderings of the same
                # arithmetic (reference autograd vs this restatement) already differ by up to ~1e-3 of the largest gradient
                close(Pg[k].grad, p_.grad, 2e-3, f"{name} oracle grad {k}", floor=gmax)
                grads[k] = {"norm": float(p_.grad.double().norm()), "full": p_.grad.detach().clone() if p_.numel() <= 4096 else None}
            o_md.update_memory(Pg, z2)
            sd = m.state_dict()
            for k in sd:
                if "running" in k or "num_batches" in k or k in ("normal_memory", "memory_ptr"):
                    close(Pg[k].detach().float(), sd[k].float(), 2e-6, f"{name} oracle state {k}", floor=1e-6)
            c.update({"loss": float(loss), "grads": grads,
                      "new_stats": {k: v.clone() for k, v in sd.items() if "running" in k or "num_batches" in k or k == "memory_ptr"},
                      "memory_rows": sd["normal_memory"][37:37 + B].clone()})
        cases.append(c)
    torch.save({"cases": cases}, os.path.join(GOLD, "md.pt"))
    print("   wrote md.pt", os.path.getsize(os.path.join(GOLD, "md.pt")) // 1024, "KiB")



def make_me():
    """M-E: the bbox visualiser's placeholder model, eval forward on a batch and on sliding windows (bbox:51-101, 328-357, 392)."""
    print("== M-E (avenue_training_script_bbox.py)")
    bbox = import_ref("avenue_training_script_bbox")
    torch.manual_seed(0)
    m = bbox.CausalAnomalyDetector().eval()
    sd = synth.synth_fill(m.state_dict(), 555)
    m.load_state_dict(sd, strict=True)
    x = synth.mb_clips(4, 8, 64, 64, 77)
    with torch.no_grad():
        s, a, f = m(x)
    frames = torch.rand(41, 3, 64, 64, generator=synth.gen(78))
    ws, wa = [], []
    with torch.no_grad():
        for st in range(0, 41 - 8, 4):                                  # bbox:392
            clip = frames[st:st + 8].permute(1, 0, 2, 3).unsqueeze(0)   # (1,3,8,64,64), bbox:397-411 layout
            s1, a1, _ = m(clip)
            ws.append(float(s1))
            wa.append(a1[0].clone())
    torch.save({"state_keys": list(sd.keys()), "scores": s.clone(), "adj": a.clone(), "feat": f.clone(), "win_scores": torch.tensor(ws),
                "win_adj": torch.stack(wa)}, os.path.join(GOLD, "me.pt"))
    print("   wrote me.pt", os.path.getsize(os.path.join(GOLD, "me.pt")) // 1024, "KiB;", len(ws), "windows")


if __name__ == "__main__":
    which = sys.argv[1:] or ["mb", "mc", "ma", "ma0", "ma_c2", "ma_traj", "md", "me"]
    os.makedirs(GOLD, exist_ok=True)
    if "mb" in which:
        make_mb()
    if "mc" in which:
        make_mc()
    if "ma" in which:
        make_ma()
    if "ma0" in which:
        make_ma0()
    if "ma_c2" in which:
        make_ma_c2()
    if "ma_traj" in which:
        make_ma_traj()
    if "md" in which:
        make_md()
    if "me" in which:
        make_me()
    print("golden fixtures written to", GOLD)
