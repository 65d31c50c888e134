"""Long-form audio (BASELINE config 3): one long recording -> sliding windows -> the batch path -> one stream.

Reference semantics (hop == window, SURVEY 8 a11): ``cut_into_windows(duration=5)`` without overlap, windows of
<= 3 s dropped, the rest padded to 5 s (src/datasets/ami/utils.py:107,163); every window is processed on its own
(own fbank edge mirroring, own LSTM state, own median-filter zero padding, vad_engine.py:204-211); the decisions are
concatenated and re-sliced per recording, ``ceil(duration / frame_shift) + 1`` frames (predict.py:447-458), then
run-length encoded (predict.py:472-490).

Extension (hop < window): overlapping windows; probabilities are stitched by taking every frame from the window
whose centre is nearest (``b200vad_stitch_center``), then threshold + median + segments run once over the stitched
stream.

Many recordings at once: ``LongFormVad(...)([wav, ...], durations)`` returns, for each recording, exactly what the call on
that recording alone returns.  The windows of all recordings are rows of one pointer table (``vad_pipeline_rows``), read in
place -- nothing is copied, a ragged last window included -- and packed into launches of ``max_rows`` rows, so a recording may
straddle two launches.  Stitching (or, for hop == window, the per-recording slice of the concatenated windows), smoothing,
segments and binarization then each run once over all recordings through stream offsets, and the host reads the segment
triples once.  Each recording's stream is cut from its own windows (``recording_offsets([d], frames of its windows)``), as the
single call does -- not by the consecutive slicing of one flat stream that ``get_segments(durations=...)`` keeps for parity
with predict.py:447-458, which shifts every later recording once a tail window has been dropped.  The single-tensor call is
the one-recording case of the same code.

SincNet -> PyanNet (``sincnet_packed``), as predict_sincnet.get_new_cuts does it: the same 5 s windows, but the tail window
is zero padded in AUDIO (samples past the recording read as 0; the SincNet InstanceNorm sees the zeros), per-window median filter, concatenation, a slice
of ``ceil(get_num_frames(16000 d)) + 1`` frames per recording (predict_sincnet.py:330-337), run-length encoding that keeps
single-frame runs and whole-second timestamps (predict_sincnet.py:348-370, 492-504).  Overlapped windows need a hop of whole
SincNet frame steps (270 samples) so that every window's frames fall on one global grid.

``binarize`` (a ``b200vad.Binarize``) replaces threshold / median / run-length segments: it runs once over the recording's
probability stream -- the stitched one for hop < window, else the concatenated window probabilities cut to the frames the
decision stream covers -- so a region that crosses a window boundary stays one region.  Intervals are then
[first * step + t0, (last + 1) * step + t0) seconds on the mode's frame grid (b200vad.binarize), clipped to the duration.
"""

from __future__ import annotations

from typing import List, Optional, Sequence, Union

import numpy as np
import torch

from .binarize import mode_step
from .host import (fbank_num_frames, get_num_frames, merge_intervals_with_buffer, recording_offsets,
                   segments_to_intervals)

SINC_STEP = 270       # samples between SincNet frames


class LongFormVad:
    def __init__(self, packed: torch.Tensor, num_layers: int = 4, window: int = 80000, hop: Optional[int] = None,
                 thr: float = 0.5, kernel: int = 49, max_rows: int = 4096, frame_shift: float = 0.01,
                 sincnet_packed: Optional[torch.Tensor] = None, binarize=None):
        self.packed, self.L, self.sinc, self.binarize = packed, num_layers, sincnet_packed, binarize
        self.window, self.hop = int(window), int(hop if hop is not None else window)
        if self.sinc is not None:
            if self.window < 991 or not (0 < self.hop <= self.window):
                raise ValueError("need window >= 991 samples (one SincNet frame) and 0 < hop <= window")
            if self.hop != self.window and self.hop % SINC_STEP:
                raise ValueError("overlapped SincNet windows need a hop that is a multiple of 270 samples (the SincNet frame step)")
        elif self.window % 160 or self.hop % 160 or not (0 < self.hop <= self.window):
            raise ValueError("window and hop must be multiples of 160 samples with 0 < hop <= window")
        self.thr, self.kernel, self.max_rows, self.fs = thr, kernel, max_rows, frame_shift

    # ---- window bookkeeping
    def _window_arrays(self, num_samples: int):
        """windows() as two int64 arrays (start_sample, valid_samples): hop == window is cut_into_windows (windows of at most
        3 / 5 of a window dropped); otherwise windows every hop samples until one reaches the end, at least one."""
        n = int(num_samples)
        if self.hop == self.window:
            s = np.arange(0, n, self.window, dtype=np.int64)
            v = np.minimum(self.window, n - s)
            keep = v > self.window * 3 // 5
            return s[keep], v[keep]
        s = np.arange(1 + max(0, -(-(n - self.window) // self.hop)), dtype=np.int64) * self.hop
        return s, np.minimum(self.window, n - s)

    def windows(self, num_samples: int):
        """[(start_sample, valid_samples)] of the rows the recording is cut into."""
        s, v = self._window_arrays(num_samples)
        return list(zip(s.tolist(), v.tolist()))

    @staticmethod
    def _check(wav, what: str) -> None:
        if not isinstance(wav, torch.Tensor) or wav.dim() != 1 or not wav.is_cuda or wav.dtype not in (torch.float32, torch.int16) \
                or not wav.is_contiguous():
            raise ValueError(f"{what} must be a contiguous 1-D float32 or int16 CUDA tensor")

    @torch.no_grad()
    def __call__(self, wav: Union[torch.Tensor, Sequence[torch.Tensor]], duration=None, *, durations=None):
        """wav: (num_samples,) float32 or int16 (16-bit PCM, read as int16 / 32768) CUDA tensor, duration in seconds (default
        num_samples / 16000).  Returns dict(prob (W, Tw), stream_dec (L,) uint8, intervals, windows).

        wav may also be a list of such recordings, all on one device and of one dtype, with ``durations`` None or a list of
        seconds (also accepted in the second position); then the result is one such dict per recording, in input order, each
        equal to the single call's on that recording.  Every recording is checked (ValueError naming its index) before any
        device work."""
        if isinstance(wav, torch.Tensor):
            if durations is not None:
                raise ValueError("durations= is for a list of recordings; pass duration= with a single tensor")
            self._check(wav, "wav")
            return self._run([wav], [duration])[0]
        if duration is not None and durations is not None:
            raise ValueError("pass the durations of a list of recordings once, as durations=")
        durations = duration if durations is None else durations
        wavs = list(wav)
        durations = [None] * len(wavs) if durations is None else list(durations)
        if len(durations) != len(wavs):
            raise ValueError(f"{len(wavs)} recordings but {len(durations)} durations")
        for i, w in enumerate(wavs):
            self._check(w, f"wavs[{i}]")
            if w.device != wavs[0].device or w.dtype != wavs[0].dtype:
                raise ValueError(f"wavs[{i}] is {w.dtype} on {w.device}, wavs[0] is {wavs[0].dtype} on {wavs[0].device}: "
                                 "one call takes recordings of one dtype on one device")
        return self._run(wavs, durations)

    def _window_outputs(self, wavs: List[torch.Tensor], rows: torch.Tensor, W: int, Tw: int):
        """prob (W, Tw) f32 and per-window decisions dec (W, Tw) u8 of every window row, in launches of max_rows rows."""
        per = min(self.max_rows, 65535)
        probs, decs = [], []
        for b0 in range(0, W, per):
            p, d, _, _, _ = torch.ops.b200vad.vad_pipeline_rows(wavs, rows[b0:b0 + per], self.window, self.packed, self.sinc,
                                                                self.L, self.thr, self.kernel)
            probs.append(p); decs.append(d)
        if not probs:
            dev = wavs[0].device
            return torch.empty((0, Tw), dtype=torch.float32, device=dev), torch.empty((0, Tw), dtype=torch.uint8, device=dev)
        if len(probs) == 1:
            return probs[0], decs[0]
        return torch.cat(probs), torch.cat(decs)

    def plan(self, num_samples: Sequence[int], durations: Sequence[float]):
        """Host bookkeeping of a call on recordings of num_samples samples and durations seconds: (wins, rows, win_off,
        frame_off, hop_frames) = each recording's windows(), the (W, 3) int64 host row table of (recording, start, valid) of all
        windows in order, the (R + 1) offsets of each recording's windows among the rows and of its stream among the stream
        frames, and the hop in frames at which the streams are cut from the windows (Tw for hop == window)."""
        sinc = self.sinc is not None
        Tw = get_num_frames(self.window) if sinc else fbank_num_frames(self.window)
        arrays = [self._window_arrays(n) for n in num_samples]
        wins = [list(zip(s.tolist(), v.tolist())) for s, v in arrays]
        rows = torch.from_numpy(np.stack([np.repeat(np.arange(len(arrays), dtype=np.int64), [len(s) for s, _ in arrays]),
                                          np.concatenate([s for s, _ in arrays]), np.concatenate([v for _, v in arrays])], axis=1))
        if self.hop == self.window:
            # reference semantics: the recording's windows concatenated, cut to ceil(d / fs) + 1 frames (predict.py:447-458)
            lens = [recording_offsets([d], len(w) * Tw, self.fs, sincnet=sinc)[1] for d, w in zip(durations, wins)]
            hop_frames = Tw
        else:
            lens = [get_num_frames(n) if sinc else fbank_num_frames(n) for n in num_samples]      # frames of the whole recording
            hop_frames = self.hop // (SINC_STEP if sinc else 160)
        win_off, frame_off = [0], [0]
        for w, n in zip(wins, lens):
            win_off.append(win_off[-1] + len(w))
            frame_off.append(frame_off[-1] + n)
        return wins, rows, win_off, frame_off, hop_frames

    def _run(self, wavs: List[torch.Tensor], durations) -> List[dict]:
        if not wavs:
            return []
        sinc = self.sinc is not None
        dev = wavs[0].device
        R = len(wavs)
        Ns = [w.numel() for w in wavs]
        durations = [n / 16000.0 if d is None else d for n, d in zip(Ns, durations)]
        Tw = get_num_frames(self.window) if sinc else fbank_num_frames(self.window)
        wins, rows, win_off, frame_off, hop_frames = self.plan(Ns, durations)
        prob, dec = self._window_outputs(wavs, rows, win_off[-1], Tw)
        # pinned and non-blocking: segments / binarize queue behind the pipeline instead of the host waiting for it here
        offsets = torch.tensor(frame_off, dtype=torch.int64).pin_memory().to(dev, non_blocking=True)
        if self.binarize is not None:
            step, t0 = mode_step(sinc, self.fs)
            f = self.binarize.frames(step)
            sp = torch.ops.b200vad.stitch_center_streams(prob, win_off, frame_off, hop_frames)
            if sp.numel() == 0:
                stream, ivs = torch.empty(0, dtype=torch.uint8, device=dev), [[] for _ in range(R)]
            else:
                stream, seg, _ = torch.ops.b200vad.binarize(sp, offsets, f["onset"], f["offset"], f["pad_onset"], f["pad_offset"],
                                                            f["min_off"], f["min_on"])
                ivs = self.binarize.intervals(seg.tolist(), R, step, t0, durations)
        else:
            min_run = 1 if sinc else 2      # the SincNet RLE keeps single-frame runs (predict_sincnet.py:348-370)
            if self.hop == self.window:     # per-window median filter, then the per-recording slice
                stream = torch.ops.b200vad.stitch_center_streams(dec, win_off, frame_off, hop_frames)
            else:                           # one median filter over each recording's stitched stream
                sp = torch.ops.b200vad.stitch_center_streams(prob, win_off, frame_off, hop_frames)
                stream = torch.ops.b200vad.threshold_median_streams(sp, frame_off, self.thr, self.kernel)
            if stream.numel() == 0:
                ivs = [[] for _ in range(R)]
            else:
                seg, _ = torch.ops.b200vad.segments(stream, offsets, min_run)
                ivs = segments_to_intervals(seg.tolist(), R, self.fs, sincnet_durations=durations if sinc else None)
            ivs = [merge_intervals_with_buffer(iv, d, 0) for iv, d in zip(ivs, durations)]
        return [{"prob": prob[win_off[r]:win_off[r + 1]], "stream_dec": stream[frame_off[r]:frame_off[r + 1]], "intervals": ivs[r],
                 "windows": wins[r]} for r in range(R)]

    def probability_stream(self, prob: torch.Tensor, num_samples: int, duration: float) -> torch.Tensor:
        """The recording's probability stream that binarization runs over: the stitched stream for hop < window, else the
        concatenated window probabilities cut to the frames the decision stream of the reference's path covers."""
        sinc = self.sinc is not None
        if self.hop == self.window:
            flat = prob.reshape(-1)
            return flat[: recording_offsets([duration], flat.numel(), self.fs, sincnet=sinc)[1]]
        L = get_num_frames(num_samples) if sinc else fbank_num_frames(num_samples)
        return torch.ops.b200vad.stitch_center(prob, self.hop // (SINC_STEP if sinc else 160), L)
