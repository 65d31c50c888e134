"""Speech regions with onset / offset hysteresis, padding and minimum durations (pyannote's ``Binarize``).

The device kernels (``b200vad_binarize``, include/b200vad.h) work in frames; this module holds the policy in seconds, validates
it on the host before any device call, and converts between the two for a mode's frame step:

  fbank path   : step = frame_shift (0.01 s), t0 = 0 (the reference's ``k * frame_shift`` time base)
  SincNet path : step = 270 / 16000 s, t0 = 496 / 16000 s (the HALF_DURATION of predict_sincnet.py:492-504, without its
                 rounding to whole seconds)

Seconds -> frames is ``round(seconds / step)``; a region of frames [s, e) is [s * step + t0, e * step + t0) seconds, the end
clipped to the recording's duration.
"""

from __future__ import annotations

import math
from typing import List, Optional, Sequence

import numpy as np

from ._lib import BinarizeParams

FBANK_T0 = 0.0
SINC_STEP = 270 / 16000
SINC_T0 = 496 / 16000
_INT32_MAX = 2 ** 31 - 1


def mode_step(sincnet: bool, frame_shift: float = 0.01):
    """(step, t0) in seconds of the fbank or the SincNet frame grid."""
    return (SINC_STEP, SINC_T0) if sincnet else (float(frame_shift), FBANK_T0)


def stream_event_seconds(frames, sincnet: bool, window: int) -> np.ndarray:
    """Timeline frames of a streaming session (b200vad_stream_events) -> seconds since the stream's first sample.

    A push that brings the stream to n samples returns the newest nf = hop / step_samples frames of the window of the last
    ``window`` samples, which starts at sample n - window; timeline frame tau of that push is window frame j = T - nf + k with
    n = (tau - k + nf) * hop / nf.  Window frame j lies at j * step + t0 seconds after the window's start, so tau lies at
    (n - window) / 16000 + j * step + t0, and the push-dependent terms cancel:

      fbank   : T = window / 160 frames of 160 samples, t0 = 0:  tau * 0.01 s.  Every newest frame lands on the stream's 10 ms grid.
      SincNet : step = 270 / 16000, t0 = 496 / 16000, T = get_num_frames(window):
                tau * 270 / 16000 + (270 * T - window + 496) / 16000 s.  get_num_frames(window) * 270 <= window - 721 (the
                receptive field is 991 samples), so the offset is negative for every window; the result is clipped at 0.
    """
    frames = np.asarray(frames, dtype=np.float64)
    if not sincnet:
        return frames * 0.01
    from .host import get_num_frames
    return np.maximum(frames * SINC_STEP + (270 * get_num_frames(int(window)) - int(window) + 496) / 16000, 0.0)


class Binarize:
    """Binarize(onset=0.5, offset=None, min_duration_on=0.0, min_duration_off=0.0, pad_onset=0.0, pad_offset=0.0).

    pyannote's names and units: thresholds on probabilities, durations in seconds.  ``offset=None`` means ``offset = onset``.
    A frame above ``onset`` starts speech, one below ``offset`` ends it, frames in between keep the state; regions are padded
    by ``pad_onset`` / ``pad_offset``, gaps shorter than ``min_duration_off`` are filled, regions shorter than
    ``min_duration_on`` are dropped.  Raises ValueError on a non-finite threshold, offset > onset or a negative duration."""

    def __init__(self, onset: float = 0.5, offset: Optional[float] = None, min_duration_on: float = 0.0,
                 min_duration_off: float = 0.0, pad_onset: float = 0.0, pad_offset: float = 0.0):
        onset = float(onset)
        offset = onset if offset is None else float(offset)
        # the kernel compares in fp32: a threshold that is finite in fp64 but not in fp32 is refused here, not by the device call
        with np.errstate(over="ignore"):
            finite = np.isfinite(np.float32(onset)) and np.isfinite(np.float32(offset))
        if not finite:
            raise ValueError("onset and offset must be finite (in float32)")
        if offset > onset:
            raise ValueError(f"offset ({offset}) must be <= onset ({onset})")
        durations = dict(min_duration_on=min_duration_on, min_duration_off=min_duration_off, pad_onset=pad_onset,
                         pad_offset=pad_offset)
        for name, v in durations.items():
            if not (math.isfinite(float(v)) and float(v) >= 0.0):
                raise ValueError(f"{name} must be a finite number of seconds >= 0, got {v}")
        self.onset, self.offset = onset, offset
        self.min_duration_on, self.min_duration_off = float(min_duration_on), float(min_duration_off)
        self.pad_onset, self.pad_offset = float(pad_onset), float(pad_offset)

    def __repr__(self):
        return (f"Binarize(onset={self.onset}, offset={self.offset}, min_duration_on={self.min_duration_on}, "
                f"min_duration_off={self.min_duration_off}, pad_onset={self.pad_onset}, pad_offset={self.pad_offset})")

    def frames(self, step: float) -> dict:
        """The policy on a grid of ``step`` seconds: onset, offset and the four counts round(seconds / step) under the kernel's
        names (pad_onset, pad_offset, min_off, min_on)."""
        if not (math.isfinite(step) and step > 0):
            raise ValueError("step must be a positive number of seconds")
        out = dict(onset=self.onset, offset=self.offset)
        for name, sec in (("pad_onset", self.pad_onset), ("pad_offset", self.pad_offset), ("min_off", self.min_duration_off),
                          ("min_on", self.min_duration_on)):
            n = round(sec / step)
            if n > _INT32_MAX:
                raise ValueError(f"{name} = {sec} s is more than 2^31 - 1 frames of {step} s")
            out[name] = int(n)
        return out

    def params(self, step: float) -> BinarizeParams:
        """The b200vad_binarize_params struct for a grid of ``step`` seconds."""
        return BinarizeParams(**self.frames(step))

    @staticmethod
    def intervals(seg_rows: Sequence[Sequence[int]], num_streams: int, step: float, t0: float,
                  durations: Optional[Sequence[float]] = None) -> List[List[List[float]]]:
        """(S, 3) triples (stream, first, last) -> per stream [[start_s, end_s], ...] with start = first * step + t0 and
        end = (last + 1) * step + t0, clipped to durations[stream] when given."""
        out: List[List[List[float]]] = [[] for _ in range(num_streams)]
        for r, a, b in seg_rows:
            end = (b + 1) * step + t0
            if durations is not None:
                end = min(end, durations[r])
            out[r].append([a * step + t0, end])
        return out
