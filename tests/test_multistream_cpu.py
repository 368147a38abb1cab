"""The host's window rule of infer.MultiStreamScorer (``infer.window_count``, the copy of ma0_tail.cu's ``stream_push``) against a
brute-force enumeration of the frames at which windows end."""
import math
import random

import pytest


def _windows_ending_in(lo, hi, T, stride):
    """Windows w (frames w*stride + [0, T)) whose last frame lies in [lo, hi)."""
    return [(f - (T - 1)) // stride for f in range(lo, hi) if f >= T - 1 and (f - (T - 1)) % stride == 0]


@pytest.mark.parametrize("T", [4, 16])
@pytest.mark.parametrize("stride", [1, 3, 4])
def test_window_count_vs_enumeration(T, stride):
    from cvad_b200.infer import window_count
    rnd = random.Random(T * 10 + stride)
    for n in (1, 2, 4, 7, 16):
        n_frames = next_window = 0
        m_max = 0
        for push in range(300):
            count = rnd.choice([0, n, rnd.randint(0, n)])
            reset = rnd.random() < 0.05
            base = 0 if reset else n_frames
            want = _windows_ending_in(base, base + count, T, stride)
            frames, n_win = window_count(n_frames, next_window, count, reset, T, stride)
            nxt = 0 if reset else next_window
            assert frames == base + count
            assert n_win == len(want), (n, push, base, count, want)
            assert want == list(range(nxt, nxt + n_win)), "the completed windows follow the next window without a gap"
            n_frames, next_window = frames, nxt + n_win
            m_max = max(m_max, n_win)
        assert m_max <= math.ceil(n / stride)
