"""Binarization without a GPU: the frame-domain reference against a literal restatement of pyannote's Binarize, its
degenerate case (plain thresholding), the seconds <-> frames conversion of b200vad.Binarize for both front ends, and the
host-side refusal of invalid policies."""
import math

import numpy as np
import pytest

import binarize_oracle as bo
from b200vad.binarize import SINC_STEP, SINC_T0, Binarize, mode_step


def _stream(g, T):
    kind = g.integers(4)
    if kind == 0:       # random walk around the thresholds
        return (0.5 + 0.08 * np.cumsum(g.standard_normal(T))).astype(np.float32)
    if kind == 1:       # uniform noise
        return g.uniform(0, 1, T).astype(np.float32)
    if kind == 2:       # runs of a few levels, thresholds included
        levels = np.array([0.2, 0.4, 0.5, 0.6, 0.8, np.nan], np.float32)
        return np.repeat(g.choice(levels, T), g.integers(1, 6, T))[:T]
    return (g.uniform(0, 1, T) > 0.5).astype(np.float32)


def test_oracle_equals_pyannote_restatement():
    g = np.random.default_rng(0)
    for _ in range(3000):
        T = int(g.integers(0, 120))
        x = _stream(g, T)
        onset = float(g.choice([0.5, 0.6, 0.7]))
        offset = float(min(onset, g.choice([0.3, 0.4, 0.5, 0.6])))
        pad_on, pad_off, min_off, min_on = (int(v) for v in g.choice([0, 0, 1, 2, 3, 7, 200], 4))
        dec, regions = bo.binarize(x, onset, offset, pad_on, pad_off, min_off, min_on)
        want = bo.pyannote_binarize(x, onset, offset, pad_on, pad_off, min_off, min_on)
        assert [tuple(r) for r in regions] == [tuple(w) for w in want], (x.tolist(), onset, offset, pad_on, pad_off, min_off, min_on)
        ref = np.zeros(T, np.uint8)
        for s, e in want:
            ref[s:e] = 1
        assert np.array_equal(dec, ref)


def test_degenerate_policy_is_thresholding():
    g = np.random.default_rng(1)
    for theta in (0.5, 0.3, 0.9):
        for _ in range(200):
            T = int(g.integers(0, 300))
            x = g.uniform(0, 1, T).astype(np.float32)
            x[x == np.float32(theta)] = 0.0
            dec, _ = bo.binarize(x, theta, theta)
            assert np.array_equal(dec, (x > np.float32(theta)).astype(np.uint8))


def test_seconds_to_frames_both_front_ends():
    b = Binarize(onset=0.7, offset=0.4, min_duration_on=0.25, min_duration_off=0.1, pad_onset=0.05, pad_offset=0.034)
    step, t0 = mode_step(False)
    assert (step, t0) == (0.01, 0.0)
    assert b.frames(step) == dict(onset=0.7, offset=0.4, pad_onset=5, pad_offset=3, min_off=10, min_on=25)
    step, t0 = mode_step(True)
    assert step == 270 / 16000 and t0 == 496 / 16000
    f = b.frames(step)
    assert (f["pad_onset"], f["pad_offset"], f["min_off"], f["min_on"]) == (
        round(0.05 / step), round(0.034 / step), round(0.1 / step), round(0.25 / step)) == (3, 2, 6, 15)
    assert Binarize(onset=0.6).offset == 0.6
    p = b.params(0.01)
    assert (p.pad_onset, p.pad_offset, p.min_off, p.min_on) == (5, 3, 10, 25) and math.isclose(p.onset, 0.7, rel_tol=1e-7)


def test_frames_to_seconds_both_front_ends():
    seg = [(0, 0, 9), (0, 20, 20), (1, 5, 99)]
    ivs = Binarize.intervals(seg, 2, 0.01, 0.0, [0.15, 0.5])
    assert ivs[0] == [[0.0, 0.1], [0.2, min(0.21, 0.15)]]
    assert ivs[1] == [[0.05, 0.5]]
    ivs = Binarize.intervals(seg, 2, SINC_STEP, SINC_T0, [10.0, 1.0])
    assert ivs[0] == [[SINC_T0, 10 * SINC_STEP + SINC_T0], [20 * SINC_STEP + SINC_T0, 21 * SINC_STEP + SINC_T0]]
    assert ivs[1] == [[5 * SINC_STEP + SINC_T0, 1.0]]


@pytest.mark.parametrize("kwargs", [
    dict(onset=0.4, offset=0.5), dict(onset=float("nan")), dict(onset=0.5, offset=float("-inf")), dict(onset=1e39),
    dict(min_duration_on=-0.01), dict(min_duration_off=-1.0), dict(pad_onset=-0.5), dict(pad_offset=float("inf")),
    dict(pad_onset=float("nan")),
])
def test_invalid_policy_raises_on_host(kwargs, monkeypatch):
    import b200vad._lib as lib

    def no_device(*a, **k):
        raise AssertionError("the device library was reached")
    monkeypatch.setattr(lib, "lib", no_device)
    with pytest.raises(ValueError):
        Binarize(**kwargs)


def test_counts_beyond_int32_raise():
    with pytest.raises(ValueError):
        Binarize(pad_onset=3e7).frames(0.01)
