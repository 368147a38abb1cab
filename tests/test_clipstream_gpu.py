"""Multi-stream sliding windows for the 3-D clip models (cvad_b200/infer.py ``MultiStreamClipScorer``, frames.cu
``cvad_streams_frame_write_u8`` / ``cvad_streams_clips_f32``): the two frame-ring kernels bit for bit against the single-video frame path
(``DeviceFrames``) and cv2, their argument checks, every stream of a ragged run against its own video scored alone for M-B, M-E and M-C,
graph reuse (including M-B's per-batch-size mask), weight updates through the graphs, and the errors."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

T, STRIDE, CAP, SIZE = 8, 4, 32, (64, 64)
INVALID = 1           # cudaErrorInvalidValue


def _completed(frames, T=T, stride=STRIDE):
    return (frames - T) // stride + 1 if frames >= T else 0


def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-12))


def _frames(shape, seed, dev):
    return torch.randint(0, 256, shape, generator=torch.Generator(device=dev).manual_seed(seed), device=dev, dtype=torch.uint8)


def _cv2():
    try:
        import cv2
        return cv2
    except ImportError:
        return None


def _model(kind, dev, gold):
    import synth
    from cvad_b200 import mb, mc, me
    if kind == "mb":
        m = mb.CausalAnomalyDetector()
        m.load_state_dict(gold("best_improved_model.pth")["model_state_dict"], strict=True)
    else:
        m = me.CausalAnomalyDetector() if kind == "me" else mc.SimpleVideoAnomalyDetector()
        m.load_state_dict(synth.synth_fill(m.state_dict(), 7 if kind == "me" else 8), strict=True)
    return m.to(dev).eval()


def _ref_clips(video, starts, rgb):
    """What the reference builds per window from a whole video: cv2 resize, BGR -> RGB (C = 3), /255, (C, T, H, W)."""
    from cvad_b200.frames import DeviceFrames
    return DeviceFrames(video, video.device).resized(SIZE).clips_f32(starts, T, rgb=rgb)


# ------------------------------------------------------------------------------------------------ 1. the kernels
@pytest.mark.parametrize("sh,sw,C", [(360, 640, 3), (48, 40, 3), (64, 64, 1)])
def test_frame_ring_kernels_vs_frame_path(dev, sh, sw, C):
    """Frame write, clip gather (with and without channel reversal; unused slots exact zeros) and cursor advance of S = 5 streams over
    several pushes with counts 0..n, resets and wrap-around: rings against DeviceFrames.resized (and cv2.resize where it imports), clips
    against clips_f32 of the same frames, bit for bit.  Source rows beyond a count hold a sentinel and leave the rings unchanged."""
    from cvad_b200.frames import DeviceFrames
    from cvad_b200.infer import window_count
    from cvad_b200.ops import _call, _ptr, _st
    cv2 = _cv2()
    S, n, cap = 5, 6, 16
    dw, dh = SIZE
    rings = _frames((S, cap, dh, dw, C), 1, dev)
    frames0 = [3, 40, 17, 0, 95]
    cursors = torch.tensor([[f, _completed(f)] for f in frames0], dtype=torch.int64, device=dev)
    schedule = [([0, 6, 3, 6, 5], [0, 0, 0, 0, 0]), ([6, 0, 6, 1, 6], [0, 1, 0, 0, 1]), ([6, 6, 6, 6, 6], [1, 0, 0, 1, 0]),
                ([2, 5, 0, 6, 6], [0, 0, 1, 0, 0]), ([6, 6, 6, 0, 6], [0, 0, 0, 0, 0]), ([5, 6, 6, 6, 3], [0, 0, 0, 0, 0])]
    wrapped = windows = 0
    for i, (counts, resets) in enumerate(schedule):
        ring_ref, cur = rings.clone(), cursors.tolist()
        src = _frames((S, n, sh, sw, C), 10 + i, dev)
        for k in range(S):
            src[k, counts[k]:] = 0xA5                                       # sentinel rows: never read
        resized = DeviceFrames(src.reshape(S * n, sh, sw, C), dev).resized(SIZE).data.reshape(S, n, dh, dw, C)
        if cv2 is not None:
            host = src.cpu().numpy()
            want = np.stack([np.stack([cv2.resize(f if C > 1 else f[..., 0], SIZE) for f in host[k]]) for k in range(S)])
            assert np.array_equal(resized.cpu().numpy(), want.reshape(resized.shape))
        push = torch.tensor([[c, r] for c, r in zip(counts, resets)], dtype=torch.int64, device=dev)
        wins = [window_count(cur[k][0], cur[k][1], counts[k], resets[k], T, STRIDE) for k in range(S)]
        m = max(nw for _, nw in wins) + 1                                   # one slot more than any stream needs: zero-filled
        for k in range(S):
            base = 0 if resets[k] else cur[k][0]
            wrapped += base % cap + counts[k] > cap
            for r in range(counts[k]):
                ring_ref[k, (base + r) % cap] = resized[k, r]
        outs = {rev: torch.full((S * m, C, T, dh, dw), float("nan"), device=dev) for rev in (0, 1)}
        st = _st()
        _call("cvad_streams_frame_write_u8", _ptr(src), S, n, sh, sw, C, _ptr(rings), cap, dh, dw, T, STRIDE, _ptr(cursors), _ptr(push), st)
        for rev, out in outs.items():
            _call("cvad_streams_clips_f32", _ptr(rings), S, cap, dh, dw, C, T, STRIDE, m, _ptr(cursors), _ptr(push), 1.0 / 255.0, rev,
                  _ptr(out), st)
        _call("cvad_streams_cursor_advance", _ptr(cursors), S, T, STRIDE, _ptr(push), st)
        torch.cuda.synchronize()
        assert torch.equal(rings, ring_ref), (counts, resets)
        for rev, out in outs.items():
            for k, (_, nw) in enumerate(wins):
                nxt = 0 if resets[k] else cur[k][1]
                for j in range(m):
                    got = out[k * m + j]
                    if j >= nw:
                        assert torch.equal(got, torch.zeros_like(got)), (k, j)
                        continue
                    idx = [((nxt + j) * STRIDE + t) % cap for t in range(T)]
                    want = DeviceFrames(ring_ref[k, idx], dev).clips_f32([0], T, rgb=bool(rev))[0]
                    assert torch.equal(got, want), (counts, resets, k, j, rev)
                    windows += 1
        nxt = [0 if resets[k] else cur[k][1] for k in range(S)]
        assert cursors.tolist() == [[fr, nxt[k] + nw] for k, (fr, nw) in enumerate(wins)]
    assert wrapped >= 3 and windows >= 10, (wrapped, windows)


# ------------------------------------------------------------------------------------------------ 2. argument checks
def test_frame_ring_kernels_reject_invalid_arguments(dev):
    from cvad_b200._lib import lib
    from cvad_b200.ops import _ptr
    L = lib()
    S, n, m, C, H, W = 2, 4, 1, 3, 20, 24
    src = torch.zeros(S * n, H, W, C, dtype=torch.uint8, device=dev)
    rings = torch.zeros(S, CAP, 16, 16, C, dtype=torch.uint8, device=dev)
    out = torch.zeros(S * m, C, T, 16, 16, device=dev)
    cursors = torch.zeros(S, 2, dtype=torch.int64, device=dev)
    push = torch.tensor([[n, 0]] * S, dtype=torch.int64, device=dev)
    calls = {
        "cvad_streams_frame_write_u8": dict(src=_ptr(src), S=S, n=n, src_h=H, src_w=W, C=C, rings=_ptr(rings), cap=CAP, dst_h=16, dst_w=16,
                                            T=T, stride=STRIDE, cursors=_ptr(cursors), push=_ptr(push), st=None),
        "cvad_streams_clips_f32": dict(rings=_ptr(rings), S=S, cap=CAP, H=16, W=16, C=C, T=T, stride=STRIDE, m=m, cursors=_ptr(cursors),
                                       push=_ptr(push), scale=1.0, rev=1, out=_ptr(out), st=None),
    }
    bad = {"src": [None], "rings": [None], "cursors": [None], "push": [None], "out": [None], "S": [0, -1], "cap": [0, -1], "T": [0, -1],
           "stride": [0, -1], "src_h": [0, -1], "src_w": [0, -1], "dst_h": [0, -1], "dst_w": [0, -1], "H": [0, -1], "W": [0, -1],
           "C": [0, 5], "n": [-1], "m": [-1]}
    tried = 0
    for name, args in calls.items():
        fn = getattr(L, name)
        assert fn(*args.values()) == 0                   # the valid call goes through
        for key, values in bad.items():
            if key not in args:
                continue
            for v in values:
                assert fn(*{**args, key: v}.values()) == INVALID, (name, key, v)
                tried += 1
        empty = "n" if "n" in args else "m"
        assert fn(*{**args, empty: 0}.values()) == 0
    torch.cuda.synchronize()
    assert tried == 23 + 19, tried


# ------------------------------------------------------------------------------------------------ 3. each stream as if alone
# per push: (n, counts of the S = 4 streams); stream RESET_STREAM starts over with a new video before push RESET_AT
SCHEDULE = [(6, [6, 3, 0, 6]), (8, [8, 8, 8, 2]), (3, [0, 3, 3, 3]), (8, [7, 8, 1, 8]), (8, [8, 0, 8, 8]), (4, [4, 4, 4, 0]),
            (8, [8, 8, 8, 8]), (8, [2, 8, 8, 5]), (5, [5, 1, 5, 4]), (8, [8, 8, 6, 8]), (8, [0, 8, 8, 8]), (2, [2, 2, 1, 1])]
RESET_AT, RESET_STREAM = 6, 1


def _camera_shape(kind):
    return (360, 640, 3) if kind in ("mb", "me") else (64, 64)


def _run_schedule(ms, kind, dev):
    """Push SCHEDULE through ``ms``; returns {(stream, video): the frames pushed of it}, {(stream, video): [(scores, w0, adj, feats), ...]} and the clips
    the scorer gathered, re-gathered by the same kernel from its rings after each push (with the cursors and descriptor of that push)."""
    from cvad_b200.ops import _call, _ptr, _st
    S = 4
    shape = _camera_shape(kind)
    C = 3 if len(shape) == 3 else 1
    pos, video = [0] * S, [0] * S
    total = [sum(c[k] for _, c in SCHEDULE) for k in range(S)]
    vids = {(k, 0): _frames((total[k],) + shape, 100 + k, dev) for k in range(S)}
    vids[(RESET_STREAM, 1)] = _frames((total[RESET_STREAM],) + shape, 110, dev)
    res = {key: [] for key in vids}
    gathered = {key: [] for key in vids}
    used = {key: 0 for key in vids}
    for i, (n, counts) in enumerate(SCHEDULE):
        resets = [0] * S
        if i == RESET_AT:
            ms.reset(RESET_STREAM)
            assert ms.n_frames[RESET_STREAM] == 0 and ms.next_window[RESET_STREAM] == 0
            resets[RESET_STREAM], video[RESET_STREAM], pos[RESET_STREAM] = 1, 1, 0
        x = _frames((S, n) + shape, 200 + i, dev)                          # rows beyond a count: other frames, never read
        where = []
        for k in range(S):
            x[k, :counts[k]] = vids[(k, video[k])][pos[k]:pos[k] + counts[k]]
            where.append(((k, video[k]), pos[k]))
        before = ms.cursors.clone() if ms.cursors is not None else torch.zeros(S, 2, dtype=torch.int64, device=dev)
        out = ms.push(x, counts)
        assert ms.cursors.tolist() == [[a, b] for a, b in zip(ms.n_frames, ms.next_window)]
        assert ms.n_frames == [p + c for (_, p), c in zip(where, counts)]
        m = max(r[0].shape[0] for r in out)
        if m:
            push = torch.tensor([[c, r] for c, r in zip(counts, resets)], dtype=torch.int64, device=dev)
            clips = torch.empty((S * m, C, T) + SIZE[::-1], device=dev)
            _call("cvad_streams_clips_f32", _ptr(ms.rings), S, ms.capacity, SIZE[1], SIZE[0], C, T, STRIDE, m, _ptr(before), _ptr(push),
                  1.0 / 255.0, int(C == 3), _ptr(clips), _st())
        for k, ((key, p), c, r) in enumerate(zip(where, counts, out)):
            s, w0 = r[0], r[1]
            assert w0 == _completed(p) and s.shape == (_completed(p + c) - _completed(p),), (k, p, c, w0, s.shape)
            res[key].append(r)
            used[key] += c
            if s.shape[0]:
                gathered[key].append(clips[k * m:k * m + s.shape[0]])
        for k in range(S):
            pos[k] += counts[k]
    return {key: v[:used[key]] for key, v in vids.items()}, res, gathered


@pytest.mark.parametrize("kind", ["mb", "me", "mc"])
def test_clipstream_matches_each_stream_alone(dev, gold, kind):
    """S = 4 ragged streams, one starting over mid-run with a new video.  For every stream and window: the window indices follow
    window_count, the clip the scorer gathered equals DeviceFrames(video).resized(size).clips_f32([w*stride], T) bit for bit, and scores,
    adjacency and features equal the model on those clips (1e-6 relative).  M-E: the common windows also equal me.score_windows_device,
    whose finite-video loop has one window fewer exactly when (F - T) % stride == 0."""
    from cvad_b200 import infer, me
    from cvad_b200.frames import DeviceFrames
    m = _model(kind, dev, gold)
    ms = infer.MultiStreamClipScorer(m, 4, clip_len=T, stride=STRIDE, capacity=CAP, size=SIZE)
    vids, res, gathered = _run_schedule(ms, kind, dev)
    for n in {k[0] for k in ms.graphs}:
        assert sum(k[0] == n for k in ms.graphs) <= math.ceil(n / STRIDE) + 1, sorted(ms.graphs)
    worst = {"scores": 0.0, "adjacency": 0.0, "features": 0.0}
    bbox_rule = set()
    for key, recs in res.items():
        F = vids[key].shape[0]
        n_win = sum(r[0].shape[0] for r in recs)
        assert n_win == _completed(F)
        starts = [w * STRIDE for w in range(n_win)]
        want_clips = _ref_clips(vids[key], starts, rgb=kind != "mc")
        assert torch.equal(torch.cat(gathered[key]), want_clips), key
        with torch.no_grad():
            want = m(want_clips)
        want = (want[0].reshape(-1), want[1], want[2]) if kind != "mc" else (want.reshape(-1),)
        for (name, i), w in zip((("scores", 0), ("adjacency", 2), ("features", 3)), want):
            worst[name] = max(worst[name], _rel(torch.cat([r[i] for r in recs]), w))
        if kind == "mc":
            assert all(r[2] is None and r[3] is None for r in recs)
        if kind == "me":
            frames_f = DeviceFrames(vids[key], dev).resized(SIZE).clips_f32([0], F)[0].permute(1, 0, 2, 3)     # (F, 3, H, W) RGB in [0, 1]
            s_ref, a_ref, f_ref = me.score_windows_device(m, frames_f, T, STRIDE)
            n_bbox = len(range(0, F - T, STRIDE))
            assert n_win - n_bbox == (1 if (F - T) % STRIDE == 0 else 0), (F, n_win, n_bbox)
            bbox_rule.add(n_win - n_bbox)
            got = [torch.cat([r[i] for r in recs])[:n_bbox] for i in (0, 2, 3)]
            for g, w in zip(got, (s_ref, a_ref, f_ref)):
                assert _rel(g, w) < 1e-6
    if kind == "me":
        assert bbox_rule == {0, 1}, "the schedule has videos on both sides of the rule"
    print(f"[clipstream {kind}] {len(ms.graphs)} graphs for {len(SCHEDULE)} pushes; max relative difference vs model(clips): "
          + ", ".join(f"{k} {v:.2e}" for k, v in worst.items() if k == "scores" or kind != "mc"))
    assert all(v < 1e-6 for v in worst.values()), worst


# ------------------------------------------------------------------------------------------------ 4. graph reuse
def test_clipstream_one_replay_whatever_the_stream_count(dev, gold):
    """The same push sizes at S = 1 and S = 8 issue the same ABI calls inside their graphs."""
    from cvad_b200 import infer
    m = _model("mb", dev, gold)
    x = _frames((8, 8, 360, 640, 3), 300, dev)
    launches = []
    for S in (1, 8):
        ms = infer.MultiStreamClipScorer(m, S)
        ms.push(x[:S])
        ms.push(x[:S])
        assert sorted(k[:2] for k in ms.graphs) == [(8, 1), (8, 2)]
        launches.append({k[:2]: g.launches for k, g in ms.graphs.items()})
    print(f"[clipstream] ABI calls per replay, S = 1: {launches[0]}, S = 8: {launches[1]}")
    assert launches[0] == launches[1]


def test_clipstream_graphs_of_different_batch_sizes_stay_valid(dev, gold):
    """M-B caches its self-loop mask for the latest batch size only.  Graphs captured at S*m = 2, 4 and 6 (and eager forwards at other
    batch sizes in between) are replayed alternately: every score still equals the model on the same clips."""
    from cvad_b200 import infer
    m = _model("mb", dev, gold)
    S = 2
    seq = _frames((S, 200, 360, 640, 3), 310, dev)
    ms = infer.MultiStreamClipScorer(m, S, capacity=CAP)
    # frames per push per stream: 8 -> 1 window (m = 1), 4 -> 1, 8 -> 2, 12 -> 3; the m = 1 / 2 / 3 graphs alternate after all are captured
    plan = [8, 8, 12, 4, 8, 12, 4, 8, 4, 12, 8, 4, 12, 8]
    pos, ms_seen, checked = 0, set(), 0
    for n in plan:
        res = ms.push(seq[:, pos:pos + n])
        pos += n
        ms_seen.add(max(r[0].shape[0] for r in res))
        for k, (s, w0, a, f) in enumerate(res):
            if not s.shape[0]:
                continue
            clips = _ref_clips(seq[k, :pos], [w * STRIDE for w in range(w0, w0 + s.shape[0])], rgb=True)
            with torch.no_grad():
                ws, wa, wf = m(clips)                                     # eager, at a batch size of its own: replaces the cached mask
            assert _rel(s, ws.reshape(-1)) < 1e-6 and _rel(a, wa) < 1e-6 and _rel(f, wf) < 1e-6, (n, k)
            checked += 1
    assert {1, 2, 3} <= ms_seen and checked >= 20
    assert len({k[1] for k in ms.graphs}) >= 3


# ------------------------------------------------------------------------------------------------ 5. weight updates
def test_clipstream_follows_weight_updates(dev, gold):
    """In-place updates of M-C's BatchNorm running statistics and of an M-B weight reach the scores through the captured graphs (no
    capture); a replaced tensor makes the scorer capture exactly once more."""
    from cvad_b200 import infer
    for kind in ("mc", "mb"):
        m = _model(kind, dev, gold)
        S, n = 3, 8
        seq = _frames((S, 6 * n) + _camera_shape(kind), 320, dev)
        ms = infer.MultiStreamClipScorer(m, S)
        ms.push(seq[:, :n])
        ms.push(seq[:, n:2 * n])
        graphs = dict(ms.graphs)
        assert len(graphs) == 2

        def push_and_check(i):
            res = ms.push(seq[:, i * n:(i + 1) * n])
            out = []
            for k, r in enumerate(res):
                s, w0 = r[0], r[1]
                clips = _ref_clips(seq[k, :(i + 1) * n], [w * STRIDE for w in range(w0, w0 + s.shape[0])], rgb=kind == "mb")
                with torch.no_grad():
                    want = m(clips)
                want = want[0].reshape(-1) if kind == "mb" else want.reshape(-1)
                assert s.shape[0] == 2 and _rel(s, want) < 1e-6, (kind, i, k, s, want)
                out.append(s)
            return torch.cat(out)
        before = push_and_check(2)
        with torch.no_grad():
            if kind == "mc":
                m.features[1].running_mean.add_(0.3)
                m.features[5].running_var.mul_(2.0)
            else:
                m.feature_extractor.conv3d_2.weight.mul_(1.5)
                m.anomaly_predictor[0].weight.mul_(0.5)
        for k in range(S):
            ms.reset(k)
        ms.push(seq[:, :n])
        ms.push(seq[:, n:2 * n])
        after = push_and_check(2)
        assert ms.graphs == graphs, "an in-place change must not capture again"
        assert not torch.equal(before, after), kind
        lin = m.classifier[6] if kind == "mc" else m.anomaly_predictor[2]
        lin.weight = torch.nn.Parameter(lin.weight.detach() * 0.5)
        push_and_check(3)
        assert len(ms.graphs) == 1 and all(g is not graphs.get(k) for k, g in ms.graphs.items())


# ------------------------------------------------------------------------------------------------ 6. errors
def test_clipstream_errors(dev, gold):
    from cvad_b200 import infer
    mb_m, mc_m = _model("mb", dev, gold), _model("mc", dev, gold)
    with pytest.raises(TypeError, match="MultiStreamClipScorer scores"):
        infer.MultiStreamClipScorer(torch.nn.Linear(2, 2).eval(), 2)
    mc_m.train()
    with pytest.raises(RuntimeError, match=r"MultiStreamClipScorer needs model\.eval\(\)"):
        infer.MultiStreamClipScorer(mc_m, 2)
    mc_m.eval()
    with pytest.raises(ValueError, match="ring capacity"):
        infer.MultiStreamClipScorer(mc_m, 2, clip_len=8, stride=4, capacity=11)
    with pytest.raises(ValueError, match="at least one stream"):
        infer.MultiStreamClipScorer(mc_m, 0)
    mc_s = infer.MultiStreamClipScorer(mc_m, 2, capacity=16)
    mb_s = infer.MultiStreamClipScorer(mb_m, 2, capacity=16)
    x1 = torch.zeros(2, 12, 64, 64, dtype=torch.uint8, device=dev)
    x3 = torch.zeros(2, 12, 64, 64, 3, dtype=torch.uint8, device=dev)
    with pytest.raises(TypeError, match="raw uint8 frames"):
        mc_s.push(x1.float())
    for bad in (torch.zeros(2, 12, 64, dtype=torch.uint8, device=dev), torch.zeros(1, 2, 12, 64, 64, 1, dtype=torch.uint8, device=dev)):
        with pytest.raises(ValueError, match=r"expected \(S, n, H, W, C\) frames"):
            mc_s.push(bad)
    with pytest.raises(ValueError, match="takes 1-channel frames, got 3"):
        mc_s.push(x3)
    for bad in (x1, x3[..., :1], torch.zeros(2, 12, 64, 64, 4, dtype=torch.uint8, device=dev)):
        with pytest.raises(ValueError, match="takes 3-channel frames"):
            mb_s.push(bad)
    with pytest.raises(ValueError, match="expected frames of 2 streams, got 3"):
        mc_s.push(torch.zeros(3, 4, 64, 64, dtype=torch.uint8, device=dev))
    for counts in ([4], [4, 4, 4], [-1, 4], [4, 13]):
        with pytest.raises(ValueError, match=r"counts must be 2 ints in \[0, 12\]"):
            mc_s.push(x1, counts)
    with pytest.raises(ValueError, match="more new frames than the ring can take"):
        mc_s.push(x1, [9, 0])
    with pytest.raises(RuntimeError):
        mc_s.push(x1.cpu(), [4, 4])
    mc_s.push(x1, [8, 0])                                   # within capacity - clip_len = 8 per stream, although n = 12 exceeds it
    assert mc_s.n_frames == [8, 0]
    mb_s.push(x3, [8, 3])
    assert mb_s.n_frames == [8, 3]
    mc_m.train()
    with pytest.raises(RuntimeError, match=r"MultiStreamClipScorer needs model\.eval\(\)"):
        mc_s.push(x1, [4, 4])
    mc_m.eval()
    with pytest.raises(IndexError):
        mc_s.reset(2)
