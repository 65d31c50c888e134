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
