"""Frame-domain reference of the binarization (include/b200vad.h, b200vad_binarize): a plain per-frame loop over one stream,
written from the contract, and a literal restatement of pyannote's Binarize (its loop, Timeline.support(collar) and the
removal of short tracks) on frame timestamps that the CPU tests hold it to.  Test infrastructure only."""
from __future__ import annotations

import numpy as np


def binarize(x, onset, offset, pad_onset=0, pad_offset=0, min_off=0, min_on=0):
    """x: one stream of float32 probabilities -> (dec uint8 (T,), [(s, e_exclusive), ...])."""
    x = np.asarray(x, dtype=np.float32)
    T = len(x)
    onset, offset = np.float32(onset), np.float32(offset)
    # 1. hysteresis
    a = np.zeros(T, np.uint8)
    state = 0
    for t in range(T):
        if x[t] > onset:
            state = 1
        elif x[t] < offset:
            state = 0
        a[t] = state
    # 2. maximal runs, padded and clipped; overlapping or touching ones merge
    regions = []
    start = None
    for t in range(T + 1):
        on = t < T and a[t]
        if on and start is None:
            start = t
        elif not on and start is not None:
            regions.append([max(0, start - pad_onset), min(T, t + pad_offset)])
            start = None
    merged = []
    for s, e in regions:
        if merged and s <= merged[-1][1]:
            merged[-1][1] = max(merged[-1][1], e)
        else:
            merged.append([s, e])
    # 3. gaps shorter than min_off are filled
    filled = []
    for s, e in merged:
        if filled and s - filled[-1][1] < min_off:
            filled[-1][1] = e
        else:
            filled.append([s, e])
    # 4. short regions are dropped; 5. raster
    out = [(s, e) for s, e in filled if e - s >= min_on]
    dec = np.zeros(T, np.uint8)
    for s, e in out:
        dec[s:e] = 1
    return dec, out


def pyannote_binarize(x, onset, offset, pad_onset=0, pad_offset=0, min_off=0, min_on=0):
    """pyannote.audio.utils.signal.Binarize.__call__ for one class, restated with frame indices as timestamps, followed by
    pyannote.core's Timeline.support(collar=min_off) and the min_duration_on filter.  The contract's two adjustments are marked:
    a region open at the last frame ends at T (pyannote: at the last timestamp, T - 1), and regions are clipped to [0, T)."""
    x = np.asarray(x, dtype=np.float32)
    T = len(x)
    if T == 0:
        return []
    onset, offset = np.float32(onset), np.float32(offset)
    timestamps = list(range(T))
    active = []
    start = timestamps[0]
    is_active = x[0] > onset
    for t, y in zip(timestamps[1:], x[1:]):
        if is_active:
            if y < offset:
                active.append((start - pad_onset, t + pad_offset))
                start = t
                is_active = False
        else:
            if y > onset:
                start = t
                is_active = True
    if is_active:
        active.append((start - pad_onset, T + pad_offset))           # adjustment: pyannote closes at t = T - 1
    active = [(max(0, s), min(T, e)) for s, e in active]             # adjustment: clipped to the stream
    if pad_offset > 0 or pad_onset > 0 or min_off > 0:
        active = _support(sorted(active), collar=min_off)
    if min_on > 0:
        active = [seg for seg in active if seg[1] - seg[0] >= min_on]
    return active


def _support(segments, collar):
    """pyannote.core Timeline.support_iter: gaps shorter than collar are filled, overlapping / touching segments merge
    (a gap of zero duration is 'no gap')."""
    if not segments:
        return []
    out = []
    new = segments[0]
    for seg in segments:
        gap = seg[0] - new[1]       # duration of the gap Segment(new.end, seg.start); <= 0: no gap
        if gap <= 0 or gap < collar:
            new = (min(new[0], seg[0]), max(new[1], seg[1]))
        else:
            out.append(new)
            new = seg
    out.append(new)
    return out
