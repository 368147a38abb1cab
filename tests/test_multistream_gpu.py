"""Multi-stream sliding-window inference (cvad_b200/infer.py ``MultiStreamScorer``, ma0_tail.cu ``cvad_streams_*``): the three ring
kernels bit for bit against a torch restatement, every stream of a ragged multi-stream run against the same stream scored alone, rows
beyond a stream's count, graph reuse, and the errors."""
import math

import pytest
import torch

from test_infer_gpu import ZeroNoise, _g, _ma0_model, _ma_model, _score_clip_by_clip, rel

pytestmark = pytest.mark.gpu

T, STRIDE = 16, 4


def _completed(frames):
    return (frames - T) // STRIDE + 1 if frames >= T else 0


# ------------------------------------------------------------------------------------------------ 1. the kernels
def test_streams_kernels_vs_torch(dev):
    """Ring write, window gather (unused slots zero) and cursor advance of S = 5 streams over several pushes with counts 0..n, resets and
    wrap-around, against a torch restatement: bit for bit (the kernels only copy)."""
    from cvad_b200.infer import window_count
    from cvad_b200.ops import _call, _ptr, _st
    S, cap, F, n = 5, 24, 6144, 8
    g = _g(21)
    rings = torch.randn(S, cap, F, generator=g).to(dev)
    frames0 = [3, 40, 17, 0, 95]               # consistent cursors: next window = windows completed so far
    cursors = torch.tensor([[f, _completed(f)] for f in frames0], dtype=torch.int64, device=dev)
    schedule = [([0, 8, 3, 8, 5], [0, 0, 0, 0, 0]), ([8, 0, 8, 1, 8], [0, 1, 0, 0, 1]), ([8, 8, 8, 8, 8], [1, 0, 0, 1, 0]),
                ([2, 7, 0, 8, 6], [0, 0, 1, 0, 0]), ([8, 8, 8, 0, 8], [0, 0, 0, 0, 0]), ([5, 8, 8, 8, 3], [0, 0, 0, 0, 0])]
    wrapped = 0
    for counts, resets in schedule:
        ring_ref, cur = rings.clone(), cursors.tolist()
        feats = torch.randn(S * n, F, generator=g).to(dev)
        for k in range(S):
            feats[k * n + counts[k]:(k + 1) * n] = float("nan")          # rows beyond the count must not be read
        push = torch.tensor([[c, r] for c, r in zip(counts, resets)], dtype=torch.int64, device=dev)
        wins = [window_count(cur[k][0], cur[k][1], counts[k], resets[k], T, STRIDE) for k in range(S)]
        m = max(nw for _, nw in wins) + 1                                  # one slot more than any stream needs: zero-filled
        for k in range(S):
            base = 0 if resets[k] else cur[k][0]
            wrapped += base % cap + counts[k] > cap
            for r in range(counts[k]):
                ring_ref[k, (base + r) % cap] = feats[k * n + r]
        want = torch.zeros(S * m, T, F, device=dev)
        for k, (_, nw) in enumerate(wins):
            nxt = 0 if resets[k] else cur[k][1]
            for j in range(nw):
                for t in range(T):
                    want[k * m + j, t] = ring_ref[k, ((nxt + j) * STRIDE + t) % cap]
        out = torch.full((S * m, T, F), float("nan"), device=dev)
        st = _st()
        _call("cvad_streams_ring_write_f32", _ptr(feats), S, n, F, _ptr(rings), cap, T, STRIDE, _ptr(cursors), _ptr(push), st)
        _call("cvad_streams_window_features_f32", _ptr(rings), S, cap, STRIDE, T, F, m, _ptr(cursors), _ptr(push), _ptr(out), st)
        _call("cvad_streams_cursor_advance", _ptr(cursors), S, T, STRIDE, _ptr(push), st)
        torch.cuda.synchronize()
        assert torch.equal(rings, ring_ref), (counts, resets)
        assert torch.equal(out, want), (counts, resets)
        nxt = [0 if resets[k] else cur[k][1] for k in range(S)]
        assert cursors.tolist() == [[fr, nxt[k] + nw] for k, (fr, nw) in enumerate(wins)]
    assert wrapped >= 3, "the schedule writes across the end of the rings"


def test_streams_kernels_reject_invalid_arguments(dev):
    from cvad_b200.ops import _call, _ptr
    S, cap, F, n, m = 2, 24, 64, 4, 1
    rings = torch.zeros(S, cap, F, device=dev)
    feats = torch.zeros(S * n, F, device=dev)
    out = torch.zeros(S * m, T, F, device=dev)
    cursors = torch.zeros(S, 2, dtype=torch.int64, device=dev)
    push = torch.zeros(S, 2, dtype=torch.int64, device=dev)
    calls = {
        "cvad_streams_ring_write_f32": dict(feats=_ptr(feats), S=S, n=n, F=F, rings=_ptr(rings), cap=cap, T=T, stride=STRIDE, cursors=_ptr(cursors),
                                            push=_ptr(push), st=None),
        "cvad_streams_window_features_f32": dict(rings=_ptr(rings), S=S, cap=cap, stride=STRIDE, T=T, F=F, m=m, cursors=_ptr(cursors),
                                                 push=_ptr(push), out=_ptr(out), st=None),
        "cvad_streams_cursor_advance": dict(cursors=_ptr(cursors), S=S, T=T, stride=STRIDE, push=_ptr(push), st=None),
    }
    bad = {"F": [6], "cap": [0, -1], "S": [0, -2], "stride": [0], "T": [0], "m": [-1], "n": [-1],
           "feats": [None], "rings": [None], "cursors": [None], "push": [None], "out": [None]}
    tried = 0
    for name, args in calls.items():
        _call(name, *args.values())                  # the valid call goes through
        for key, values in bad.items():
            if key not in args:
                continue
            for v in values:
                with pytest.raises(RuntimeError, match=name):
                    _call(name, *{**args, key: v}.values())
                tried += 1
    torch.cuda.synchronize()
    assert tried == 30


# ------------------------------------------------------------------------------------------------ 2-4. the scorer against each stream alone
H, W, CAP = 64, 96, 24
# per push: (n, counts of the S = 4 streams); every count <= CAP - T = 8; stream 2 starts over before push RESET_AT with a new video
SCHEDULE = [(5, [5, 3, 0, 5]), (8, [8, 8, 8, 2]), (3, [0, 3, 3, 3]), (8, [7, 8, 1, 8]), (8, [8, 0, 8, 8]), (4, [4, 4, 4, 0]),
            (8, [8, 8, 8, 8]), (8, [2, 8, 8, 5]), (4, [4, 1, 4, 4]), (8, [8, 8, 6, 8]), (8, [0, 8, 8, 8]), (8, [8, 8, 8, 8]),
            (2, [2, 2, 2, 1]), (8, [8, 5, 8, 8]), (8, [8, 8, 8, 0])]
RESET_AT, RESET_STREAM = 7, 2


def _videos():
    """Frames of every stream's videos: stream k's first video, and the second video of the stream that starts over."""
    S = 4
    total = [sum(c[k] for _, c in SCHEDULE) for k in range(S)]
    vids = {(k, 0): torch.randint(0, 256, (total[k], 1, H, W), generator=_g(30 + k), dtype=torch.uint8) for k in range(S)}
    vids[(RESET_STREAM, 1)] = torch.randint(0, 256, (total[RESET_STREAM], 1, H, W), generator=_g(40), dtype=torch.uint8)
    return vids


def _pushes(vids, dev, garbage_seed, fp32=False):
    """The schedule as (frames (S, n, 1, H, W), counts, reset stream or None, [(video, first frame) per stream]); the rows beyond a
    stream's count hold random finite frames drawn from ``garbage_seed``."""
    S = 4
    pos = {k: 0 for k in range(S)}
    video = {k: 0 for k in range(S)}
    g = _g(garbage_seed)
    out = []
    for i, (n, counts) in enumerate(SCHEDULE):
        reset = None
        if i == RESET_AT:
            reset = RESET_STREAM
            video[reset], pos[reset] = 1, 0
        x = torch.randint(0, 256, (S, n, 1, H, W), generator=g, dtype=torch.uint8)
        where = []
        for k in range(S):
            x[k, :counts[k]] = vids[(k, video[k])][pos[k]:pos[k] + counts[k]]
            where.append((video[k], pos[k]))
            pos[k] += counts[k]
        if fp32:
            x = (x.float() - 0.5) / 0.5
            for k in range(S):                          # the discarded rows: any finite values, not only normalised pixels
                x[k, counts[k]:] = torch.randn(n - counts[k], 1, H, W, generator=g) * 3.0
        out.append((x.to(dev), counts, reset, where))
    return out


@pytest.mark.parametrize("kind", ["ma", "ma0"])
def test_multistream_matches_each_stream_alone(dev, gold, kind):
    """S = 4 ragged streams (per-push counts 0..n, one stream starts over mid-run with a new video): after every push each stream's ring
    rows equal a fresh FrozenBackbone over that stream's frames bit for bit and the device cursors equal the host mirrors; at the end every
    video's scores equal clip-by-clip scoring (2e-5, the graphed single-stream bound) and the fp32 model (1e-3).  No (n, m) pair is
    captured twice, and the graph count stays within ceil(n / stride) + 1 per push size."""
    from cvad_b200 import infer
    m = _ma_model(dev) if kind == "ma" else _ma0_model(dev, gold)
    m.noise = ZeroNoise()
    m.set_precision("bf16")
    S = 4
    vids_cpu = _videos()
    vids = {key: v.to(dev) for key, v in vids_cpu.items()}
    ms = infer.MultiStreamScorer(m, S, clip_len=T, stride=STRIDE, capacity=CAP)
    ref_fz = infer.FrozenBackbone(m.backbone)
    ring_ref = torch.zeros(S, CAP, 6144, device=dev)
    scores = {key: [] for key in vids}
    seen = {}
    for x, counts, reset, where in _pushes(vids_cpu, dev, 50):
        if reset is not None:
            ms.reset(reset)
            assert ms.n_frames[reset] == 0 and ms.next_window[reset] == 0
        res = ms.push(x, counts)
        n = x.shape[1]
        mm = 0
        for k, ((s, w0), c, (v, p)) in enumerate(zip(res, counts, where)):
            assert w0 == _completed(p) and s.shape == (_completed(p + c) - _completed(p),), (k, p, c, w0, s.shape)
            mm = max(mm, s.shape[0])
            scores[(k, v)].append(s)
            if c:
                f = ref_fz(vids[(k, v)][p:p + c])
                for r in range(c):
                    ring_ref[k, (p + r) % CAP] = f[r]
        assert torch.equal(ms.rings, ring_ref)
        assert ms.cursors.tolist() == [[a, b] for a, b in zip(ms.n_frames, ms.next_window)]
        assert ms.n_frames == [p + c for (_, p), c in zip(where, counts)]
        key = (n, mm, H, W, torch.uint8)
        assert key in ms.graphs
        if key in seen:
            assert ms.graphs[key] is seen[key], f"{key} captured again"
        seen[key] = ms.graphs[key]
    assert len(ms.graphs) <= len({(k[0], k[1]) for k in seen})
    for n in {k[0] for k in ms.graphs}:
        assert sum(k[0] == n for k in ms.graphs) <= math.ceil(n / STRIDE) + 1
    worst, worst32 = 0.0, 0.0
    for (k, v), ss in scores.items():
        got = torch.cat(ss)
        n_win = got.shape[0]
        if n_win == 0:
            continue
        seq = vids[(k, v)]
        want = _score_clip_by_clip(m, seq, T, STRIDE, n_win)
        with torch.no_grad():
            m.set_precision("fp32")
            want32 = m(torch.stack([seq[w * STRIDE: w * STRIDE + T] for w in range(n_win)]))["anomaly_scores"]
            m.set_precision("bf16")
        worst, worst32 = max(worst, rel(got, want)), max(worst32, rel(got, want32))
    print(f"[multistream {kind}] {len(ms.graphs)} graphs for {len(SCHEDULE)} pushes: vs clip by clip {worst:.2e} (2e-5), vs fp32 "
          f"{worst32:.2e} (1e-3)")
    assert worst < 2e-5 and worst32 < 1e-3


@pytest.mark.parametrize("fp32", [False, True])
def test_rows_beyond_counts_do_not_matter(dev, fp32):
    """The same schedule twice with different finite frames beyond every count: the rings come out bit-identical."""
    from cvad_b200 import infer
    m = _ma_model(dev)
    m.noise = ZeroNoise()
    vids = _videos()
    rings = []
    for garbage in (60, 61):
        ms = infer.MultiStreamScorer(m, 4, clip_len=T, stride=STRIDE, capacity=CAP)
        for x, counts, reset, _ in _pushes(vids, dev, garbage, fp32):
            if reset is not None:
                ms.reset(reset)
            ms.push(x, counts)
        rings.append(ms.rings.clone())
    assert torch.equal(rings[0], rings[1])


def test_one_replay_whatever_the_stream_count(dev):
    """The same push sizes at S = 1 and S = 8 issue the same ABI calls inside their graphs: one replay per push for any S."""
    from cvad_b200 import infer
    m = _ma_model(dev)
    m.noise = ZeroNoise()
    x = torch.randint(0, 256, (8, 8, 1, H, W), generator=_g(70), dtype=torch.uint8).to(dev)
    launches = []
    for S in (1, 8):
        ms = infer.MultiStreamScorer(m, S, clip_len=T, stride=STRIDE, capacity=CAP)
        ms.push(x[:S])
        ms.push(x[:S])
        assert sorted(k[:2] for k in ms.graphs) == [(8, 0), (8, 1)]
        launches.append({k[:2]: g.launches for k, g in ms.graphs.items()})
    print(f"[multistream] ABI calls per replay, S = 1: {launches[0]}, S = 8: {launches[1]}")
    assert launches[0] == launches[1]


def test_multistream_follows_weight_updates(dev):
    """An in-place change reaches every stream through the captured graphs (no capture); a replaced tensor makes the scorer capture again.
    After each change one push of 16 frames per stream completes a window made of frames pushed after the change: its ring rows are
    checked against a fresh FrozenBackbone bit for bit and its score against clip-by-clip scoring."""
    from cvad_b200 import infer
    m = _ma_model(dev)
    m.noise = ZeroNoise()
    S, n, cap = 3, 16, 40
    seq = torch.randint(0, 256, (S, 5 * n, 1, H, W), generator=_g(80), dtype=torch.uint8).to(dev)
    ms = infer.MultiStreamScorer(m, S, clip_len=T, stride=STRIDE, capacity=cap)
    ms.push(seq[:, :n])
    ms.push(seq[:, n:2 * n])
    graphs = dict(ms.graphs)
    assert len(graphs) == 2

    def push_and_check(i):
        res = ms.push(seq[:, i * n:(i + 1) * n])
        fz = infer.FrozenBackbone(m.backbone)
        for k, (s, w0) in enumerate(res):
            f = fz(seq[k, i * n:(i + 1) * n])
            for r in range(n):
                assert torch.equal(ms.rings[k, (i * n + r) % cap], f[r]), (i, k, r)
            last = w0 + s.shape[0] - 1
            assert last * STRIDE == i * n
            want = _score_clip_by_clip(m, seq[k, i * n:], T, STRIDE, 1)
            assert rel(s[-1:], want) < 2e-5, (i, k, s, want)
    with torch.no_grad():
        m.backbone.layer2[0].weight.mul_(1.25)
        m.backbone.layer3[4].running_var.mul_(1.5)
        m.direct_classifier[0].weight.mul_(0.75)
    push_and_check(2)
    assert ms.graphs == graphs, "an in-place change must not capture again"
    m.backbone.layer1[0].weight = torch.nn.Parameter(m.backbone.layer1[0].weight.detach() * 0.5)
    push_and_check(3)
    assert len(ms.graphs) == 1 and all(g is not graphs.get(k) for k, g in ms.graphs.items())


# ------------------------------------------------------------------------------------------------ 5. errors
def test_multistream_errors(dev):
    """The checks GraphedStreamingScorer also makes raise the same types and messages; a wrong stream count and counts outside [0, n] or
    above capacity - clip_len raise ValueError."""
    from cvad_b200 import infer
    m = _ma_model(dev)
    m.train()
    for args in ((m, 2), (m,)):
        cls = infer.MultiStreamScorer if len(args) == 2 else infer.GraphedStreamingScorer
        with pytest.raises(RuntimeError, match=r"needs model\.eval\(\)"):
            cls(*args)
    m.eval()
    with pytest.raises(ValueError, match="ring capacity"):
        infer.MultiStreamScorer(m, 2, clip_len=16, stride=4, capacity=19)
    ms = infer.MultiStreamScorer(m, 2, clip_len=16, stride=4, capacity=24)
    gs = infer.GraphedStreamingScorer(m, clip_len=16, stride=4, capacity=24)
    for bad_multi, bad_single in ((torch.zeros(2, 9, 1, H, W, dtype=torch.uint8, device=dev), torch.zeros(9, 1, H, W, dtype=torch.uint8, device=dev)),
                                  (torch.zeros(2, 4, 1, H, W, dtype=torch.uint8), torch.zeros(4, 1, H, W, dtype=torch.uint8))):
        with pytest.raises((RuntimeError, ValueError)) as e_multi:
            ms.push(bad_multi)
        with pytest.raises((RuntimeError, ValueError)) as e_single:
            gs.push(bad_single)
        assert (type(e_multi.value), str(e_multi.value)) == (type(e_single.value), str(e_single.value))
    with pytest.raises(ValueError, match=r"expected \(S, n, 1, H, W\) frames"):
        ms.push(torch.zeros(4, 1, H, W, dtype=torch.uint8, device=dev))
    x = torch.zeros(2, 12, 1, H, W, dtype=torch.uint8, device=dev)
    with pytest.raises(ValueError, match="expected frames of 2 streams, got 3"):
        ms.push(torch.zeros(3, 4, 1, H, W, dtype=torch.uint8, device=dev))
    for counts in ([4], [4, 4, 4], [-1, 4], [4, 13]):
        with pytest.raises(ValueError, match=r"counts must be 2 ints in \[0, 12\]"):
            ms.push(x, counts)
    with pytest.raises(ValueError, match="more new frames than the ring can take"):
        ms.push(x, [9, 0])
    ms.push(x, [8, 0])                                  # within capacity - clip_len per stream, although n = 12 exceeds it
    assert ms.n_frames == [8, 0]
    m.train()
    with pytest.raises(RuntimeError, match=r"MultiStreamScorer needs model\.eval\(\)"):
        ms.push(x, [4, 4])
    m.eval()
    with pytest.raises(IndexError):
        ms.reset(2)
