"""CPU tests of the streaming speech events: the online reference in stream_events_oracle against the offline binarization
reference (final pairs and the earliest-certainty emission frame of every event) over seeded streams, policies and chunkings;
the seconds conversion of both front ends; and argument refusal of the new C entries, which needs no device."""
import ctypes as C

import numpy as np
import pytest

import binarize_oracle as bo
import stream_events_oracle as so

EINVAL = -1


def _stream(g, T):
    kind = g.integers(5)
    if kind == 0:
        x = 0.5 + 0.15 * np.cumsum(g.standard_normal(T))
    elif kind == 1:
        x = np.repeat(g.uniform(0, 1, T), g.integers(1, 12, T))[:T]
    elif kind == 2:
        x = np.repeat(g.choice(np.array([0.0, 1.0, 0.5, np.nan, np.inf, -np.inf]), T), g.integers(1, 6, T))[:T]
    elif kind == 3:
        x = (np.arange(T) % 2 == 0).astype(np.float64)
    else:
        x = g.uniform(0, 1, T)
    return x.astype(np.float32)


def _policy(g, T):
    onset = float(g.choice([0.5, 0.6, 0.7]))
    offset = float(g.choice([onset, 0.4, 0.3]))
    big = T + int(g.integers(0, 5))
    cnt = lambda: int(g.choice([0, 1, 2, 3, 7, int(g.integers(0, 40)), big]))
    return (onset, offset, cnt(), cnt(), cnt(), cnt())


def _chunks(g, T):
    """random chunk sizes covering T: mostly small, sometimes up to 2049, varying between calls"""
    out, n = [], 0
    while n < T:
        k = int(g.choice([1, 1, 2, 31, 32, 33, int(g.integers(1, 300)), int(g.integers(1, 2050))]))
        out.append(k)
        n += k
    return out


def _run(x, policy, chunks):
    ref = so.OnlineRegions(*policy)
    events, n = [], 0
    for k in chunks:
        ev = ref.push(x[n:n + k])
        assert len(ev) <= min(k, len(x) - n)               # at most one event per frame
        events += ev
        n += k
    last = ref.end()
    assert len(last) <= 1
    return events + last


@pytest.mark.parametrize("block", range(10))
def test_online_reference_matches_offline(block):
    """300 draws per block: final pairs equal bo.binarize on the whole timeline; each emission frame equals the
    earliest-certainty definition (checked on timelines short enough for the quadratic offline search)."""
    g = np.random.default_rng(1000 + block)
    for _ in range(300):
        T = int(g.choice([int(g.integers(0, 40)), int(g.integers(0, 160)), int(g.integers(0, 5000))]))
        x = _stream(g, T)
        policy = _policy(g, T)
        events = _run(x, policy, _chunks(g, T))
        assert so.pairs(events) == bo.binarize(x, *policy)[1], (T, policy)
        frames = [e[1] for e in events]
        assert frames == sorted(frames) and [e[2] for e in events] == sorted(e[2] for e in events)
        if T <= 160:
            assert events == so.offline_emission_frames(x, policy), (T, policy, x.tolist())


def test_policy_switch_pairs_equal_per_segment_reference():
    g = np.random.default_rng(5)
    for _ in range(200):
        T1, T2 = int(g.integers(0, 300)), int(g.integers(0, 300))
        x = _stream(g, T1 + T2)
        p1, p2 = _policy(g, T1), _policy(g, T2)
        a = _run(x[:T1], p1, _chunks(g, T1))
        b = _run(x[T1:], p2, _chunks(g, T2))
        assert so.pairs(a) == bo.binarize(x[:T1], *p1)[1]
        assert so.pairs(b) == bo.binarize(x[T1:], *p2)[1]


def test_alternating_input_fills_nf_plus_one():
    """min_on = 0 and gap_break = 1: every frame of 1 0 1 0 ... emits, and an odd chunk ending on a 1 adds the end of stream"""
    for nf in (1, 2, 31, 32, 33, 2049):
        x = (np.arange(nf) % 2 == 0).astype(np.float32)
        ref = so.OnlineRegions(0.5, 0.5, 0, 0, 0, 0)
        ev = ref.push(x) + ref.end()
        assert len(ev) == nf + (nf % 2)


def test_seconds_conversion():
    from b200vad.binarize import stream_event_seconds
    from b200vad.host import get_num_frames
    f = np.array([0, 1, 7, 100, 360000])
    assert np.array_equal(stream_event_seconds(f, False, 80000), f * 0.01)
    for W in (991, 16000, 80000, 80270):
        Ts = get_num_frames(W)
        want = np.maximum(f * 270 / 16000 + (270 * Ts - W + 496) / 16000, 0)
        got = stream_event_seconds(f, True, W)
        assert np.allclose(got, want, rtol=0, atol=1e-9)
        assert (270 * Ts - W + 496) < 0 and got[0] == 0.0
        # timeline frame tau is window frame j = Ts - nf + k of the push that brought the stream to n samples: its time from
        # the stream's start is (n - W) / 16000 + j * 270 / 16000 + 496 / 16000
        nf = 3
        for tau in (5, 40, 1000):
            k = tau % nf
            n = (tau - k + nf) * 270
            if n < W:
                continue
            direct = (n - W) / 16000 + (Ts - nf + k) * 270 / 16000 + 496 / 16000
            assert abs(stream_event_seconds([tau], True, W)[0] - max(direct, 0.0)) < 1e-12


def test_new_entries_refuse_bad_arguments_without_a_device():
    import b200vad
    from b200vad import _lib
    L = b200vad.lib()
    P = _lib.BinarizeParams
    state = (C.c_int64 * 10)()
    ev = (C.c_int64 * 8)()
    counts = (C.c_int32 * 2)()
    prob = (C.c_float * 4)()
    good = P(0.5, 0.5, 0, 0, 0, 0)
    for p in (P(0.4, 0.5, 0, 0, 0, 0), P(float("nan"), 0.5, 0, 0, 0, 0), P(0.5, float("inf"), 0, 0, 0, 0), P(0.5, 0.5, -1, 0, 0, 0),
              P(0.5, 0.5, 0, 0, 0, -1)):
        assert L.b200vad_regions_step(prob, 2, 2, 2, p, state, None, ev, counts, 3, None) == EINVAL
    assert L.b200vad_regions_step(prob, 2, 2, 2, None, state, None, ev, counts, 3, None) == EINVAL
    assert L.b200vad_regions_step(prob, -1, 2, 2, good, state, None, ev, counts, 3, None) == EINVAL
    assert L.b200vad_regions_step(prob, 2, -1, 2, good, state, None, ev, counts, 3, None) == EINVAL
    assert L.b200vad_regions_step(prob, 2, 2, 1, good, state, None, ev, counts, 3, None) == EINVAL      # row stride < nf
    assert L.b200vad_regions_step(prob, 2, 2, 2, good, state, None, ev, counts, -1, None) == EINVAL
    assert L.b200vad_regions_step(None, 2, 2, 2, good, state, None, ev, counts, 3, None) == EINVAL
    assert L.b200vad_regions_step(prob, 2, 2, 2, good, None, None, ev, counts, 3, None) == EINVAL
    assert L.b200vad_regions_step(prob, 2, 2, 2, good, state, None, None, counts, 3, None) == EINVAL
    assert L.b200vad_regions_step(prob, 2, 2, 2, good, state, None, ev, None, 3, None) == EINVAL
    assert L.b200vad_regions_step(None, 0, 0, 0, good, None, None, None, None, 0, None) == 0       # nothing to do
    n = C.c_int64(0)
    assert L.b200vad_stream_set_events(None, good) == EINVAL
    assert L.b200vad_stream_end(None, (C.c_int32 * 1)(0), 1) == EINVAL
    assert L.b200vad_stream_events(None, None, 0, C.byref(n)) == EINVAL
