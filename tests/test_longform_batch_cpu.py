"""CPU tests of LongFormVad over many recordings: the host bookkeeping of the list call (windows, row table, window and stream
offsets) against R single-recording windows() results, argument refusal before any device work, and the new C entries."""
import math
import os

import numpy as np
import pytest
import torch

from b200vad.host import cut_into_windows, fbank_num_frames, get_num_frames, recording_offsets

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# 2 s (no reference window), 1 window, 3.9 s tail kept, 2 s tail dropped, shorter than one window, 991 samples, 0, 10 min
LENGTHS = [32000, 80000, 302400, 272000, 20000, 991, 0, 9_600_000, 80001, 128000]


def _lf(hop, sinc):
    import b200vad
    window = 80000
    if hop is not None and sinc:
        hop = 270 * 120
    return b200vad.LongFormVad(None, 4, window=window, hop=hop, sincnet_packed=torch.zeros(1) if sinc else None)


@pytest.mark.parametrize("sinc", [False, True])
@pytest.mark.parametrize("hop", [None, 40000, 16000])
def test_plan_matches_single_recordings(hop, sinc):
    lf = _lf(hop, sinc)
    rng = np.random.default_rng(7)
    lengths = LENGTHS + [int(x) for x in rng.integers(0, 3_000_000, 30)]
    durations = [n / 16000.0 if i % 3 else n / 16000.0 + 0.37 for i, n in enumerate(lengths)]     # explicit durations too
    wins, rows, win_off, frame_off, hop_frames = lf.plan(lengths, durations)
    Tw = get_num_frames(80000) if sinc else fbank_num_frames(80000)
    table = np.asarray(rows, dtype=np.int64).reshape(-1, 3)
    assert len(wins) == len(lengths) and len(win_off) == len(frame_off) == len(lengths) + 1
    assert win_off[0] == frame_off[0] == 0 and table.shape[0] == win_off[-1]
    for r, (n, d) in enumerate(zip(lengths, durations)):
        single = lf.windows(n)
        assert wins[r] == single
        sl = table[win_off[r]:win_off[r + 1]]
        assert [(int(s), int(v)) for _, s, v in sl] == single and (sl[:, 0] == r).all()
        assert ((sl[:, 1] >= 0) & (sl[:, 1] + sl[:, 2] <= n) & (sl[:, 2] <= lf.window)).all()   # rows stay inside their recording
        L = frame_off[r + 1] - frame_off[r]
        if lf.hop == lf.window:
            assert hop_frames == Tw
            # the single call's slice of its own windows' concatenated frames
            assert L == recording_offsets([d], len(single) * Tw, lf.fs, sincnet=sinc)[1] <= len(single) * Tw
            want = min(math.ceil(get_num_frames(16000 * d)) + 1 if sinc else math.ceil(d / 0.01) + 1, len(single) * Tw)
            assert L == want
        else:
            assert hop_frames == lf.hop // (270 if sinc else 160)
            assert L == (get_num_frames(n) if sinc else fbank_num_frames(n))
            assert len(single) >= 1


def _sliding_windows(num_samples, window, hop):
    """The overlapped cut as a plain loop: windows every hop samples until one reaches the end, at least one."""
    out, s = [], 0
    while True:
        out.append((s, min(window, num_samples - s)))
        if s + window >= num_samples:
            break
        s += hop
    return out


@pytest.mark.parametrize("window,hop", [(80000, 80000), (80000, 40000), (80000, 16000), (80000, 32400), (16000, 16000),
                                        (16000, 8000), (1600, 160)])
def test_windows_match_the_reference_cut(window, hop):
    """windows() is computed with numpy; it equals cut_into_windows (hop == window: windows of at most 3 / 5 of a window dropped)
    and the sliding loop (hop < window) at every length around a window or hop edge."""
    import b200vad
    lf = b200vad.LongFormVad(None, 4, window=window, hop=hop, sincnet_packed=torch.zeros(1) if hop % 160 else None)
    rng = np.random.default_rng(window + hop)
    edges = [k * m + d for m in (window, hop, window * 3 // 5) for k in range(0, 5) for d in (-1, 0, 1)]
    for n in sorted({x for x in edges + [int(v) for v in rng.integers(0, 40 * window, 200)] if x >= 0}):
        got = lf.windows(n)
        want = cut_into_windows(n, window, min_keep=window * 3 // 5) if hop == window else _sliding_windows(n, window, hop)
        assert got == want, n
        assert all(type(x) is int for w in got for x in w)


def test_durations_keyword():
    """The list form takes durations= (or the durations in the second position), never both; a single tensor takes duration=."""
    lf = _lf(40000, False)
    assert lf([], durations=None) == [] and lf([], durations=[]) == [] and lf([], []) == []
    with pytest.raises(ValueError, match="durations"):
        lf([torch.zeros(16000)] * 2, durations=[1.0])
    with pytest.raises(ValueError, match="once"):
        lf([], [1.0], durations=[1.0])
    with pytest.raises(ValueError, match="single tensor"):
        lf(torch.zeros(16000), durations=[1.0])
    with pytest.raises(ValueError, match=r"wavs\[0\]"):
        lf([torch.zeros(16000)], durations=[1.0])                  # the keyword reaches the per-recording checks


def test_plan_does_not_shift_after_a_dropped_tail():
    """A dropped tail window shortens that recording's stream only: the next recording's stream starts where its own frames do,
    unlike the consecutive slicing of one flat stream (predict.py:447-458)."""
    lf = _lf(None, False)
    lengths = [272000, 80000]                           # 17 s: 3 windows, 2 s tail dropped; then exactly one window
    wins, _, win_off, frame_off, _ = lf.plan(lengths, [17.0, 5.0])
    assert win_off == [0, 3, 4]
    assert frame_off == [0, 1500, 2000]                 # 17 s wants 1701 frames, its 3 windows hold 1500; 5 s wants 501 of 500
    flat = recording_offsets([17.0, 5.0], 2000, 0.01)
    assert flat == [0, 1701, 2000]                      # the flat slicing would start recording 1 inside it


def test_refusals_name_the_recording_before_any_device_work():
    lf = _lf(40000, False)
    with pytest.raises(ValueError, match=r"wavs\[0\]"):
        lf([torch.zeros(16000)])                        # not on a CUDA device
    with pytest.raises(ValueError, match=r"wavs\[0\]"):
        lf([torch.zeros(2, 16000)])
    with pytest.raises(ValueError, match=r"wavs\[0\]"):
        lf([torch.zeros(16000, dtype=torch.float64)])
    with pytest.raises(ValueError, match=r"wavs\[0\]"):
        lf([torch.zeros(32000)[::2]])
    with pytest.raises(ValueError, match="durations"):
        lf([torch.zeros(16000)] * 2, [1.0])
    with pytest.raises(ValueError, match="wav must be"):
        lf(torch.zeros(16000))
    assert lf([]) == []


def test_new_entries_are_declared_and_exported():
    import b200vad
    from b200vad import _lib
    header = open(os.path.join(ROOT, "include", "b200vad.h")).read()
    for name in ("b200vad_pipeline_rows", "b200vad_stitch_center_streams", "b200vad_threshold_median_streams"):
        assert name in _lib.PROTOTYPES
        assert f"B200VAD_API int {name}(" in header
        assert hasattr(b200vad.lib(), name)
    for op in ("vad_pipeline_rows", "stitch_center_streams", "threshold_median_streams"):
        assert hasattr(torch.ops.b200vad, op)


def test_new_entries_refuse_bad_arguments_without_a_device():
    import b200vad
    L = b200vad.lib()
    assert L.b200vad_stitch_center_streams(None, 2, None, None, 1, 10, 5, 10, None, None) == -1          # elem_bytes
    assert L.b200vad_stitch_center_streams(None, 4, None, None, 65536, 10, 5, 10, None, None) == -1      # R > 65535
    assert L.b200vad_stitch_center_streams(None, 4, None, None, 1, 10, 11, 10, None, None) == -1         # hop > Tw
    assert L.b200vad_stitch_center_streams(None, 4, None, None, 1, 10, 5, 10, None, None) == -1          # null pointers
    assert L.b200vad_stitch_center_streams(None, 4, None, None, 0, 10, 5, 0, None, None) == 0            # nothing to do
    assert L.b200vad_threshold_median_streams(None, None, 65536, 10, 0.5, 49, None, None) == -1
    assert L.b200vad_threshold_median_streams(None, None, 2, 10, 0.5, 49, None, None) == -1
    assert L.b200vad_threshold_median_streams(None, None, 0, 10, 0.5, 49, None, None) == 0
    assert L.b200vad_pipeline_rows(None, None, 4, None, 0, None, 65536, 80000, 0.5, 49, None, None, None, None, None, None, 0,
                                   None, 0, None) == -1
    assert L.b200vad_pipeline_rows(None, 1, 4, None, 0, None, 1, 990, 0.5, 49, None, None, None, None, None, None, 0,
                                   None, 0, None) == -1                                                  # SincNet N < 991
    assert L.b200vad_pipeline_rows(None, None, 4, None, 0, None, 3, 80000, 0.5, 49, None, None, None, None, None, None, 0,
                                   None, 0, None) == -1                                                  # null table
    bad = b200vad._lib.BinarizeParams(0.4, 0.6, 0, 0, 0, 0)                                              # offset > onset
    assert L.b200vad_pipeline_rows(None, None, 4, None, 0, None, 3, 80000, 0.5, 49, bad, None, None, None, None, None, 0,
                                   None, 0, None) == -1
