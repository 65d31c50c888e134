"""Per-frame online reference of the streaming speech events (include/b200vad.h, b200vad_regions_step), written from the
contract, and the offline definitions of each event's emission frame that the CPU tests hold it to.  Test infrastructure only."""
from __future__ import annotations

import numpy as np

import binarize_oracle as bo


class OnlineRegions:
    """One stream.  push(x) / end() -> [(kind, frame, emitted_at)]: kind 1 = start, 0 = end; frame is the region's first frame
    (start) or its exclusive end (end); emitted_at is the timeline frame whose arrival made the event certain, or T (the
    timeline length) for the event of an end of stream."""

    def __init__(self, onset, offset, pad_onset=0, pad_offset=0, min_off=0, min_on=0):
        self.onset, self.offset = np.float32(onset), np.float32(offset)
        self.pad_onset, self.pad_offset, self.min_on = int(pad_onset), int(pad_offset), int(min_on)
        self.gap_break = int(pad_onset) + int(pad_offset) + max(int(min_off), 1)
        self.reset()

    def reset(self):
        self.h = 0            # hysteresis state after the last frame
        self.last_end = -1    # end of the last region of the open group
        self.gs = -1          # start of the open group, -1: none
        self.emitted = False  # the open group's start was emitted
        self.t = 0            # frames seen

    def _passes(self, t):
        ge = t + 1 if self.h else self.last_end
        return min(t + 1, ge + self.pad_offset) - max(0, self.gs - self.pad_onset) >= self.min_on

    def push(self, x):
        out = []
        for v in np.asarray(x, dtype=np.float32):
            t = self.t
            prev = self.h
            if v > self.onset:
                self.h = 1
            elif v < self.offset:
                self.h = 0
            if self.h and not prev:                  # a region starts; it opens a group unless it joins the open one
                if self.gs < 0:
                    self.gs, self.emitted = t, False
            elif prev and not self.h:                # a region ends
                self.last_end = t
            if self.gs >= 0 and not self.emitted and self._passes(t):
                self.emitted = True
                out.append((1, max(0, self.gs - self.pad_onset), t))
            if self.gs >= 0 and not self.h and t - self.last_end + 1 >= self.gap_break:
                if self.emitted:                     # no later onset can join the group
                    out.append((0, self.last_end + self.pad_offset, t))
                self.gs = -1
            self.t += 1
        return out

    def end(self):
        """End of stream: the open group closes at T with clipping; the state is reset."""
        out = []
        T = self.t
        if self.gs >= 0 and self.emitted:
            ge = T if self.h else self.last_end
            out.append((0, min(T, ge + self.pad_offset), T))
        self.reset()
        return out


def pairs(events):
    """[(kind, frame, ...)] of one stream -> [(s, e)]"""
    out, s = [], None
    for ev in events:
        if ev[0] == 1:
            assert s is None, events
            s = ev[1]
        else:
            assert s is not None, events
            out.append((s, ev[1]))
            s = None
    assert s is None, events
    return out


def offline_emission_frames(x, policy):
    """The earliest-certainty definitions through the offline reference, for the regions bo.binarize finds on x:
    start(s) at the first t whose prefix x[:t+1] has a region starting at s; end(e) of region [s, e) at the first t such that
    x[:t+1] followed by max(min_on, 1) frames of +inf has the region [s, e) and another one after it (the +inf run either joins
    the group or survives on its own).  -> [(kind, frame, t)] in emission order; an end that no frame makes certain is the end
    of stream's, reported at T."""
    x = np.asarray(x, dtype=np.float32)
    T = len(x)
    tail = np.full(max(policy[5], 1), np.inf, np.float32)
    _, regions = bo.binarize(x, *policy)

    def closed(t, s, e):
        r = [tuple(v) for v in bo.binarize(np.concatenate([x[:t + 1], tail]), *policy)[1]]
        return (s, e) in r[:-1]

    out = []
    t = 0
    for s, e in regions:
        while s not in [r[0] for r in bo.binarize(x[:t + 1], *policy)[1]]:
            t += 1
        out.append((1, s, t))
        while t < T and not closed(t, s, e):
            t += 1
        out.append((0, e, t))
    return out
