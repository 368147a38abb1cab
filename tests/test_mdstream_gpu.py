"""Multi-stream sliding windows for M-D (cvad_b200/infer.py ``MultiStreamAutoEncoderScorer``, md_kernels.cu ``cvad_streams_md_scores_f32``):
the score kernel against a torch restatement and against ``cvad_memory_score_f32``, its argument checks, the golden M-D scores, every stream
of a ragged run against itself alone and against ``md.calculate_anomaly_scores``, each frame encoded once, rows beyond the counts, weight and
memory-bank updates through the graphs, and the errors.

The encoder's 2048 -> 64 layer adds its split-K partial sums atomically, so two runs of the same batch may differ in the last bits: the
projection rings and the scores are compared to a tight tolerance, the frame rings and cursors bit for bit."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

T, STRIDE, CAP = 8, 4, 32
E, D = 64 * 64, 64
INVALID = 1           # cudaErrorInvalidValue


def _completed(frames, T=T, stride=STRIDE):
    return (frames - T) // stride + 1 if frames >= T else 0


def _rel(a, b, floor=1e-6):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).abs().max() / max(float(b.abs().max()), floor)) if b.numel() else 0.0


def _frames(shape, seed, dev):
    """M-D input frames in [0.001, 0.999] (tests/synth.md_clips' range)."""
    return torch.rand(shape, generator=torch.Generator(device=dev).manual_seed(seed), device=dev) * 0.998 + 0.001


def _model(dev, gold, idx=1):
    """The M-D model of md.pt case idx (as test_md_eval_parity builds it): memory_ptr = 37, so the memory term is live."""
    from cvad_b200.md import VideoAutoEncoder
    from test_oracle_golden import md_reference_order, md_state_like, md_synth_state
    c = gold("md.pt")["cases"][idx]
    m = VideoAutoEncoder()
    m.load_state_dict(md_state_like(md_reference_order(md_synth_state(c["seed"]), c["state_keys"]), c["seed"]), strict=True)
    return m.to(dev).eval(), c


def _eager(m, video, w0, nw, dev):
    """calculate_anomaly_scores on the clips of windows [w0, w0 + nw) of one stream's frames (F, 1, 64, 64)."""
    from cvad_b200 import md
    clips = torch.stack([video[w * STRIDE:w * STRIDE + T] for w in range(w0, w0 + nw)])
    s, _, r, mem = md.calculate_anomaly_scores(m, [(clips, np.zeros(nw))], device=dev)
    return [torch.from_numpy(v) for v in (s, r, mem)]


# ------------------------------------------------------------------------------------------------ 1. the kernel
def test_md_scores_kernel_vs_torch(dev):
    """S = 5 streams over several pushes with counts 0..n, resets and wrap-around, m one larger than any stream needs, and the kernel called
    at several memory fill counts before each cursor advance: recon_err against an fp64 restatement over the ring rows (1e-6), mem_score
    bit for bit against cvad_memory_score_f32 at the same fill count (exact zeros below 10 rows), score = 0.7 recon + 0.3 mem as torch
    rounds it, unused slots exact zeros."""
    from cvad_b200.infer import window_count
    from cvad_b200.ops import _call, _ptr, _st
    S, n, cap, rows = 5, 6, 16, 500
    g = torch.Generator(device=dev).manual_seed(3)
    rings = torch.rand((S, cap, E), device=dev, generator=g)
    memory = torch.randn((rows, D), device=dev, generator=g)
    frames0 = [3, 40, 17, 0, 95]
    cursors = torch.tensor([[f, _completed(f)] for f in frames0], dtype=torch.int64, device=dev)
    schedule = [([0, 6, 3, 6, 5], [0, 0, 0, 0, 0]), ([6, 0, 6, 1, 6], [0, 1, 0, 0, 1]), ([6, 6, 6, 6, 6], [1, 0, 0, 1, 0]),
                ([2, 5, 0, 6, 6], [0, 0, 1, 0, 0]), ([6, 6, 6, 0, 6], [0, 0, 0, 0, 0]), ([5, 6, 6, 6, 3], [0, 0, 0, 0, 0])]
    wrapped = windows = 0
    worst = 0.0
    for i, (counts, resets) in enumerate(schedule):
        ring_ref, cur = rings.clone(), cursors.tolist()
        src = torch.rand((S * n, E), device=dev, generator=g)
        push = torch.tensor([[c, r] for c, r in zip(counts, resets)], dtype=torch.int64, device=dev)
        wins = [window_count(cur[k][0], cur[k][1], counts[k], resets[k], T, STRIDE) for k in range(S)]
        m = max(nw for _, nw in wins) + 1
        for k in range(S):
            base = 0 if resets[k] else cur[k][0]
            wrapped += base % cap + counts[k] > cap
            for r in range(counts[k]):
                ring_ref[k, (base + r) % cap] = src[k * n + r]
        recon = torch.rand((S * m, E), device=dev, generator=g)
        z = torch.randn((S * m, D), device=dev, generator=g)
        st = _st()
        _call("cvad_streams_ring_write_f32", _ptr(src), S, n, E, _ptr(rings), cap, T, STRIDE, _ptr(cursors), _ptr(push), st)
        for ptr in (0, 9, 10, 37, 500, 700):
            mp = torch.tensor([ptr], dtype=torch.int64, device=dev)
            out = [torch.full((S * m,), float("nan"), device=dev) for _ in range(3)]
            _call("cvad_streams_md_scores_f32", _ptr(rings), S, cap, E, T, STRIDE, m, _ptr(cursors), _ptr(push), _ptr(recon), _ptr(z),
                  _ptr(memory), rows, _ptr(mp), D, *map(_ptr, out), st)
            filled = min(ptr, rows)
            want_mem = torch.zeros(S * m, device=dev)
            if filled >= 10:
                _call("cvad_memory_score_f32", _ptr(z), _ptr(memory), S * m, filled, D, _ptr(want_mem), st)
            torch.cuda.synchronize()
            score, rerr, mscore = out
            for k, (_, nw) in enumerate(wins):
                nxt = 0 if resets[k] else cur[k][1]
                for j in range(m):
                    s = k * m + j
                    if j >= nw:
                        assert float(score[s]) == 0.0 and float(rerr[s]) == 0.0 and float(mscore[s]) == 0.0, (k, j, ptr)
                        assert not (score[s].signbit() or rerr[s].signbit() or mscore[s].signbit())
                        continue
                    idx = [((nxt + j) * STRIDE + t) % cap for t in range(T)]
                    want = float(((recon[s].double() - ring_ref[k, idx].double()) ** 2).mean())
                    worst = max(worst, abs(float(rerr[s]) - want) / want)
                    assert abs(float(rerr[s]) - want) <= 1e-6 * want, (k, j, float(rerr[s]), want)
                    assert torch.equal(mscore[s], want_mem[s]), (k, j, ptr, float(mscore[s]), float(want_mem[s]))
                    if filled < 10:
                        assert float(mscore[s]) == 0.0
                    windows += ptr == 0
            used = torch.tensor([j < nw for _, nw in wins for j in range(m)], device=dev)
            assert torch.equal(score[used], 0.7 * rerr[used] + 0.3 * mscore[used]), ptr
        _call("cvad_streams_cursor_advance", _ptr(cursors), S, T, STRIDE, _ptr(push), st)
        torch.cuda.synchronize()
        assert torch.equal(rings, ring_ref)
        nxt = [0 if resets[k] else cur[k][1] for k in range(S)]
        assert cursors.tolist() == [[fr, nxt[k] + nw] for k, (fr, nw) in enumerate(wins)]
    print(f"[mdstream kernel] {windows} windows, max relative recon_err difference vs fp64 {worst:.2e}")
    assert wrapped >= 3 and windows >= 10, (wrapped, windows)


# ------------------------------------------------------------------------------------------------ 2. argument checks
def test_md_scores_kernel_rejects_invalid_arguments(dev):
    from cvad_b200._lib import lib
    from cvad_b200.ops import _ptr
    fn = lib().cvad_streams_md_scores_f32
    S, m, rows = 2, 2, 500
    rings = torch.rand(S, CAP, E, device=dev)
    cursors = torch.tensor([[T + STRIDE, 0]] * S, dtype=torch.int64, device=dev)
    push = torch.tensor([[0, 0]] * S, dtype=torch.int64, device=dev)
    recon, z = torch.rand(S * m, E, device=dev), torch.randn(S * m, D, device=dev)
    memory, mp = torch.randn(rows, D, device=dev), torch.tensor([37], dtype=torch.int64, device=dev)
    outs = [torch.full((S * m,), 7.0, device=dev) for _ in range(3)]
    args = dict(rings=_ptr(rings), S=S, cap=CAP, E=E, T=T, stride=STRIDE, m=m, cursors=_ptr(cursors), push=_ptr(push), recon=_ptr(recon),
                z=_ptr(z), memory=_ptr(memory), rows=rows, mp=_ptr(mp), D=D, score=_ptr(outs[0]), recon_err=_ptr(outs[1]),
                mem_score=_ptr(outs[2]), st=None)
    bad = {k: [None] for k in ("rings", "cursors", "push", "recon", "z", "memory", "mp", "score", "recon_err", "mem_score")}
    bad.update({"E": [0, -4, 6], "S": [0, -1], "T": [0, -1], "stride": [0, -1], "cap": [0, -1], "D": [0, -1], "rows": [0, -1], "m": [-1]})
    bad["rings"].append(_ptr(rings) + 4)
    bad["recon"].append(_ptr(recon) + 4)
    tried = 0
    for key, values in bad.items():
        for v in values:
            assert fn(*{**args, key: v}.values()) == INVALID, (key, v)
            tried += 1
    assert fn(*{**args, "m": 0}.values()) == 0
    torch.cuda.synchronize()
    assert all(torch.equal(o, torch.full_like(o, 7.0)) for o in outs), "a rejected call wrote its outputs"
    assert fn(*args.values()) == 0                              # the valid call goes through
    torch.cuda.synchronize()
    assert all(bool(torch.isfinite(o).all()) and not torch.equal(o, torch.full_like(o, 7.0)) for o in outs)
    assert tried == 12 + 3 + 2 * 6 + 1, tried


# ------------------------------------------------------------------------------------------------ 3. golden anchor
@pytest.mark.parametrize("idx", [0, 1])
def test_mdstream_matches_golden(dev, gold, idx):
    """The md.pt eval cases pushed as B streams of one clip each: window 0 of every stream gives the fixture's combined score and memory
    score (cad1:545-552) to 2e-5 relative."""
    import synth
    from cvad_b200 import infer
    m, c = _model(dev, gold, idx)
    x = synth.md_clips(c["B"], c["T"], seed=c["xseed"]).to(dev)
    ms = infer.MultiStreamAutoEncoderScorer(m, c["B"], clip_len=c["T"], stride=STRIDE, capacity=2 * c["T"])
    res = ms.push(x)
    assert all(w0 == 0 and s.shape == (1,) for s, w0, _, _ in res)
    s = torch.cat([r[0] for r in res])
    mem = torch.cat([r[3] for r in res])
    assert float(mem.abs().max()) > 0
    assert _rel(s, c["combined"]) < 2e-5, (s, c["combined"])
    assert _rel(mem, c["anomaly_score"]) < 2e-5, (mem, c["anomaly_score"])
    assert torch.equal(s, 0.7 * torch.cat([r[2] for r in res]) + 0.3 * mem)


# ------------------------------------------------------------------------------------------------ 4. each stream alone and eager
# per push: (n, counts of the S = 4 streams); stream RESET_STREAM starts over with a new video before push RESET_AT
SCHEDULE = [(6, [6, 3, 0, 6]), (8, [8, 8, 8, 2]), (3, [0, 3, 3, 3]), (8, [7, 8, 1, 8]), (8, [8, 0, 8, 8]), (4, [4, 4, 4, 0]),
            (8, [8, 8, 8, 8]), (8, [2, 8, 8, 5]), (5, [5, 1, 5, 4]), (8, [8, 8, 6, 8]), (8, [0, 8, 8, 8]), (2, [2, 2, 1, 1])]
RESET_AT, RESET_STREAM = 6, 1


def _run_schedule(ms, dev, alone=None, seed=0):
    """Push SCHEDULE through ``ms`` (and each stream's frames through ``alone[k]``, an S = 1 scorer, when given).  Returns the videos
    {(stream, video): frames pushed} and the records {(stream, video): [(scores, w0, recon, mem), ...]} of ms (and of alone)."""
    S = 4
    pos, video = [0] * S, [0] * S
    total = [sum(c[k] for _, c in SCHEDULE) for k in range(S)]
    vids = {(k, 0): _frames((total[k], 1, 64, 64), 100 + k, dev) for k in range(S)}
    vids[(RESET_STREAM, 1)] = _frames((total[RESET_STREAM], 1, 64, 64), 110, dev)
    res = {key: [] for key in vids}
    res_alone = {key: [] for key in vids}
    used = {key: 0 for key in vids}
    for i, (n, counts) in enumerate(SCHEDULE):
        if i == RESET_AT:
            ms.reset(RESET_STREAM)
            if alone is not None:
                alone[RESET_STREAM].reset(0)
            assert ms.n_frames[RESET_STREAM] == 0 and ms.next_window[RESET_STREAM] == 0
            video[RESET_STREAM], pos[RESET_STREAM] = 1, 0
        x = _frames((S, n, 1, 64, 64), 200 + 1000 * seed + i, dev)          # rows beyond a count: other frames, never kept
        where = []
        for k in range(S):
            x[k, :counts[k]] = vids[(k, video[k])][pos[k]:pos[k] + counts[k]]
            where.append(((k, video[k]), pos[k]))
        out = ms.push(x, counts)
        assert ms.cursors.tolist() == [[a, b] for a, b in zip(ms.n_frames, ms.next_window)]
        assert ms.n_frames == [p + c for (_, p), c in zip(where, counts)]
        for k, ((key, p), c, r) in enumerate(zip(where, counts, out)):
            s, w0 = r[0], r[1]
            assert w0 == _completed(p) and all(t.shape == (_completed(p + c) - _completed(p),) for t in (r[0], r[2], r[3])), (k, p, c, w0)
            res[key].append(r)
            used[key] += c
            if alone is not None:
                [ra] = alone[k].push(x[k:k + 1], [c])
                assert ra[1] == w0
                res_alone[key].append(ra)
        for k in range(S):
            pos[k] += counts[k]
    return {key: v[:used[key]] for key, v in vids.items()}, res, res_alone


def test_mdstream_matches_each_stream_alone_and_eager(dev, gold):
    """S = 4 ragged streams, one starting over mid-run with a new video.  Every stream's window indices follow window_count; its scores,
    reconstruction errors and memory scores equal those of the same stream in an S = 1 scorer (1e-6 relative) and those of
    md.calculate_anomaly_scores on its window clips (2e-5)."""
    from cvad_b200 import infer
    m, _ = _model(dev, gold)
    ms = infer.MultiStreamAutoEncoderScorer(m, 4, clip_len=T, stride=STRIDE, capacity=CAP)
    alone = [infer.MultiStreamAutoEncoderScorer(m, 1, clip_len=T, stride=STRIDE, capacity=CAP) for _ in range(4)]
    vids, res, res_alone = _run_schedule(ms, dev, alone)
    for n in {k[0] for k in ms.graphs}:
        assert sum(k[0] == n for k in ms.graphs) <= math.ceil(n / STRIDE) + 1, sorted(ms.graphs)
    worst_alone, worst_eager = [0.0] * 3, [0.0] * 3
    for key, recs in res.items():
        F = vids[key].shape[0]
        n_win = sum(r[0].shape[0] for r in recs)
        assert n_win == _completed(F)
        got = [torch.cat([r[i] for r in recs]) for i in (0, 2, 3)]
        solo = [torch.cat([r[i] for r in res_alone[key]]) for i in (0, 2, 3)]
        want = _eager(m, vids[key], 0, n_win, dev)
        for i in range(3):
            worst_alone[i] = max(worst_alone[i], _rel(got[i], solo[i]))
            worst_eager[i] = max(worst_eager[i], _rel(got[i], want[i]))
        assert float(got[2].abs().min()) > 0, "the memory term is live"
    names = ("scores", "recon", "mem")
    print(f"[mdstream] {len(ms.graphs)} graphs for {len(SCHEDULE)} pushes; max relative difference vs S = 1: "
          + ", ".join(f"{k} {v:.2e}" for k, v in zip(names, worst_alone)) + "; vs calculate_anomaly_scores: "
          + ", ".join(f"{k} {v:.2e}" for k, v in zip(names, worst_eager)))
    assert all(v <= 1e-6 for v in worst_alone), worst_alone
    assert all(v <= 2e-5 for v in worst_eager), worst_eager


# ------------------------------------------------------------------------------------------------ 5. encoded once
def test_mdstream_encodes_each_frame_once(dev, gold):
    """Over a whole run the projection ring holds, for every kept frame, its row of linear_act(encode_frames(x)) with x the push's S*n
    frames as one batch (the same batch: the 2048 -> 64 layer splits its reduction by batch size), and the frame ring the frame itself.
    The graphs issue the same ABI calls at S = 1 and S = 8 for equal (n, m)."""
    from cvad_b200 import infer, ops
    m, _ = _model(dev, gold)
    lstm = m.temporal_encoder
    S, n = 3, 4
    ms = infer.MultiStreamAutoEncoderScorer(m, S, clip_len=T, stride=STRIDE, capacity=CAP)
    worst = spread = 0.0
    for i in range(12):
        x = _frames((S, n, 1, 64, 64), 400 + i, dev)
        base = ms.n_frames
        ms.push(x)
        with torch.no_grad():
            flat = x.reshape(S * n, 1, 64, 64)
            refs = [ops.linear_act(m.encode_frames(flat), lstm.weight_ih_l0, lstm.bias_ih_l0) for _ in range(2)]
        spread = max(spread, _rel(refs[0], refs[1]))
        for k in range(S):
            idx = [(base[k] + r) % CAP for r in range(n)]
            worst = max(worst, _rel(ms.rings[k, idx], refs[0][k * n:(k + 1) * n]))
            assert torch.equal(ms.frame_rings[k, idx], x[k].reshape(n, E))
    print(f"[mdstream] projection ring vs linear_act(encode_frames(x)): max relative difference {worst:.2e} (two eager runs: {spread:.2e})")
    assert worst <= 1e-5, worst
    launches = []
    xs = _frames((8, 8, 1, 64, 64), 450, dev)
    for S in (1, 8):
        ms = infer.MultiStreamAutoEncoderScorer(m, S)
        ms.push(xs[:S])
        ms.push(xs[:S])
        assert sorted(ms.graphs) == [(8, 1), (8, 2)]
        launches.append({k: g.launches for k, g in ms.graphs.items()})
    print(f"[mdstream] ABI calls per replay, S = 1: {launches[0]}, S = 8: {launches[1]}")
    assert launches[0] == launches[1]


# ------------------------------------------------------------------------------------------------ 6. rows beyond the counts
def test_mdstream_ignores_rows_beyond_counts(dev, gold):
    """The ragged schedule twice, with different finite frames beyond every count: the frame rings and cursors are bit-identical, the
    projection rings and every score agree to the last-bit spread of the encoder's split-K sums."""
    from cvad_b200 import infer
    m, _ = _model(dev, gold)
    runs = []
    for seed in (0, 1):
        ms = infer.MultiStreamAutoEncoderScorer(m, 4, clip_len=T, stride=STRIDE, capacity=CAP)
        _, res, _ = _run_schedule(ms, dev, seed=seed)
        runs.append((ms, res))
    (a, ra), (b, rb) = runs
    assert torch.equal(a.frame_rings, b.frame_rings) and torch.equal(a.cursors, b.cursors)
    worst = _rel(a.rings, b.rings)
    for key in ra:
        for x, y in zip(ra[key], rb[key]):
            assert x[1] == y[1]
            for i in (0, 2, 3):
                worst = max(worst, _rel(x[i], y[i]))
    print(f"[mdstream] other frames beyond the counts: max relative difference {worst:.2e}")
    assert worst <= 1e-5, worst


# ------------------------------------------------------------------------------------------------ 7. updates through the graphs
def test_mdstream_follows_weight_and_memory_updates(dev, gold):
    """In-place updates of encoder, decoder and LSTM weights and of BatchNorm running statistics reach the scores through the captured
    graphs; update_memory on a model whose bank starts empty turns the memory term from exact zeros into the ops.memory_score values once
    10 rows are filled, without a capture; a replaced parameter makes the scorer capture exactly once more."""
    from cvad_b200 import infer, ops
    m, _ = _model(dev, gold)
    S, n = 3, 8
    seq = _frames((S, 2 * n, 1, 64, 64), 500, dev)
    ms = infer.MultiStreamAutoEncoderScorer(m, S)

    def run():
        for k in range(S):
            ms.reset(k)
        ms.push(seq[:, :n])
        res = ms.push(seq[:, n:])
        out = []
        for k, (s, w0, r, mem) in enumerate(res):
            assert w0 == 1 and s.shape == (2,)
            want = _eager(m, seq[k], w0, 2, dev)
            for g_, w_ in zip((s, r, mem), want):
                assert _rel(g_, w_) <= 2e-5, (k, g_, w_)
            out.append(torch.stack([s, r, mem]))
        return torch.stack(out)

    before = run()
    graphs = dict(ms.graphs)
    assert sorted(graphs) == [(8, 1), (8, 2)]
    with torch.no_grad():
        m.encoder[0].weight.mul_(1.1)
        m.encoder[4].running_var.mul_(1.5)
        m.decoder[3].weight.mul_(0.9)
        m.decoder[7].running_mean.add_(0.05)
        m.temporal_encoder.weight_hh_l0.mul_(0.8)
        m.temporal_encoder.weight_ih_l0.mul_(1.2)
    after = run()
    assert ms.graphs == graphs, "an in-place change must not capture again"
    assert not torch.equal(before, after)

    with torch.no_grad():
        m.normal_memory.zero_()
        m.memory_ptr.zero_()
    m._ptr_host = None
    bank = torch.randn(11, D, device=dev)
    for rows, live in ((0, False), (6, False), (5, True)):
        if rows:
            m.update_memory(bank[:rows] if m._ptr() == 0 else bank[6:6 + rows])
        for k in range(S):
            ms.reset(k)
        ms.push(seq[:, :n])
        res = ms.push(seq[:, n:])
        mem = torch.cat([r[3] for r in res])
        if not live:
            assert torch.equal(mem, torch.zeros_like(mem)), rows
            continue
        assert m._ptr() == 11
        with torch.no_grad():
            clips = torch.stack([seq[k, w * STRIDE:w * STRIDE + T] for k in range(S) for w in (1, 2)])
            want = ops.memory_score(m.encode_sequence(clips)[0], m.normal_memory, m._ptr())
        assert float(mem.abs().min()) > 0 and _rel(mem, want) <= 2e-5, (mem, want)
    assert ms.graphs == graphs, "update_memory must not capture again"

    lin = m.decoder[0]
    lin.weight = torch.nn.Parameter(lin.weight.detach() * 0.5)
    for k in range(S):
        ms.reset(k)
    ms.push(seq[:, :n])
    assert list(ms.graphs) == [(8, 1)] and ms.graphs[(8, 1)] is not graphs[(8, 1)]
    res = ms.push(seq[:, n:])
    assert len(ms.graphs) == 2
    for k, (s, w0, _, _) in enumerate(res):
        assert _rel(s, _eager(m, seq[k], w0, 2, dev)[0]) <= 2e-5


# ------------------------------------------------------------------------------------------------ 8. errors
def test_mdstream_errors(dev, gold):
    from cvad_b200 import infer
    m, _ = _model(dev, gold)
    with pytest.raises(TypeError, match="MultiStreamAutoEncoderScorer scores md.VideoAutoEncoder"):
        infer.MultiStreamAutoEncoderScorer(torch.nn.Linear(2, 2).to(dev).eval(), 2)
    m.train()
    with pytest.raises(RuntimeError, match=r"MultiStreamAutoEncoderScorer needs model\.eval\(\)"):
        infer.MultiStreamAutoEncoderScorer(m, 2)
    m.eval()
    with pytest.raises(ValueError, match="ring capacity"):
        infer.MultiStreamAutoEncoderScorer(m, 2, clip_len=8, stride=4, capacity=11)
    with pytest.raises(ValueError, match="at least one stream"):
        infer.MultiStreamAutoEncoderScorer(m, 0)
    ms = infer.MultiStreamAutoEncoderScorer(m, 2, capacity=16)
    x = _frames((2, 12, 1, 64, 64), 600, dev)
    for bad in (x.double(), (x * 255).to(torch.uint8), x.half()):
        with pytest.raises(TypeError, match="float32 frames"):
            ms.push(bad)
    for bad in (x[:, :, :, :32, :32], x.expand(2, 12, 3, 64, 64), x[:, :, 0, 0], x[:, :, 0, :, :48], x.unsqueeze(0)):
        with pytest.raises(ValueError, match=r"expected \(S, n, 1, 64, 64\)"):
            ms.push(bad)
    with pytest.raises(ValueError, match="expected frames of 2 streams, got 3"):
        ms.push(_frames((3, 4, 1, 64, 64), 601, dev))
    for counts in ([4], [4, 4, 4], [-1, 4], [4, 13]):
        with pytest.raises(ValueError, match=r"counts must be 2 ints in \[0, 12\]"):
            ms.push(x, counts)
    with pytest.raises(ValueError, match="more new frames than the ring can take"):
        ms.push(x, [9, 0])
    with pytest.raises(RuntimeError):
        ms.push(x.cpu(), [4, 4])
    ms.push(x, [8, 0])                                      # within capacity - clip_len = 8 per stream, although n = 12 exceeds it
    assert ms.n_frames == [8, 0]
    res = ms.push(x[:, :, 0], [4, 3])                       # (S, n, 64, 64) frames
    assert ms.n_frames == [12, 3] and res[0][1] == 1 and res[0][0].shape == (1,) and res[1][0].shape == (0,)
    m.train()
    with pytest.raises(RuntimeError, match=r"MultiStreamAutoEncoderScorer needs model\.eval\(\)"):
        ms.push(x, [4, 4])
    m.eval()
    with pytest.raises(IndexError):
        ms.reset(2)
