"""Long-form audio (BASELINE config 3): one long recording -> sliding windows -> the batch path -> one stream.

Reference semantics (hop == window, SURVEY 8 a11): ``cut_into_windows(duration=5)`` without overlap, windows of
<= 3 s dropped, the rest padded to 5 s (src/datasets/ami/utils.py:107,163); every window is processed on its own
(own fbank edge mirroring, own LSTM state, own median-filter zero padding, vad_engine.py:204-211); the decisions are
concatenated and re-sliced per recording, ``ceil(duration / frame_shift) + 1`` frames (predict.py:447-458), then
run-length encoded (predict.py:472-490).

Extension (hop < window): overlapping windows; probabilities are stitched by taking every frame from the window
whose centre is nearest (``b200vad_stitch_center``), then threshold + median + segments run once over the stitched
stream.  Windows are rows of an ``as_strided`` view of the waveform: nothing is copied.

SincNet -> PyanNet (``sincnet_packed``), as predict_sincnet.get_new_cuts does it: the same 5 s windows, but the tail window
is zero padded in AUDIO (the SincNet InstanceNorm sees the zeros; no lens), per-window median filter, concatenation, a slice
of ``ceil(get_num_frames(16000 d)) + 1`` frames per recording (predict_sincnet.py:330-337), run-length encoding that keeps
single-frame runs and whole-second timestamps (predict_sincnet.py:348-370, 492-504).  Overlapped windows need a hop of whole
SincNet frame steps (270 samples) so that every window's frames fall on one global grid.

``binarize`` (a ``b200vad.Binarize``) replaces threshold / median / run-length segments: it runs once over the recording's
probability stream -- the stitched one for hop < window, else the concatenated window probabilities cut to the frames the
decision stream covers -- so a region that crosses a window boundary stays one region.  Intervals are then
[first * step + t0, (last + 1) * step + t0) seconds on the mode's frame grid (b200vad.binarize), clipped to the duration.
"""

from __future__ import annotations

from typing import Optional

import torch

from .binarize import mode_step
from .host import (cut_into_windows, fbank_num_frames, get_num_frames, merge_intervals_with_buffer, recording_offsets,
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
    def windows(self, num_samples: int):
        """[(start_sample, valid_samples)] of the rows the recording is cut into."""
        if self.hop == self.window:
            return cut_into_windows(num_samples, self.window, min_keep=self.window * 3 // 5)
        out, s = [], 0
        while True:
            n = min(self.window, num_samples - s)
            out.append((s, n))
            if s + self.window >= num_samples:
                break
            s += self.hop
        return out

    def _rows(self, wav: torch.Tensor, wins):
        """(rows, window) view of wav (row stride = hop) + per-row valid lengths; only the ragged tail is copied."""
        N = wav.numel()
        full = [w for w in wins if w[1] == self.window]
        rows = torch.as_strided(wav, (len(full), self.window), (self.hop, 1)) if full else wav.new_empty((0, self.window))
        lens = torch.full((len(wins),), self.window, dtype=torch.int32, device=wav.device)
        if len(full) != len(wins):                      # last window is short: pad it into its own row
            s, n = wins[-1]
            tail = wav.new_zeros((1, self.window))
            tail[0, :n] = wav[s:s + n]
            lens[-1] = n
            return rows, tail, lens
        return rows, None, lens

    @torch.no_grad()
    def __call__(self, wav: torch.Tensor, duration: Optional[float] = None):
        """wav: (num_samples,) float32 CUDA tensor.  Returns dict(prob (W, Tw), stream_dec (L,) uint8, intervals)."""
        if wav.dim() != 1 or not wav.is_cuda or wav.dtype != torch.float32 or not wav.is_contiguous():
            raise ValueError("wav must be a contiguous 1-D float32 CUDA tensor")
        N = wav.numel()
        duration = N / 16000.0 if duration is None else duration
        wins = self.windows(N)
        rows, tail, lens = self._rows(wav, wins)
        sinc = self.sinc is not None
        Tw = get_num_frames(self.window) if sinc else fbank_num_frames(self.window)

        def run(r, lens):
            if sinc:            # the tail row is zero padded audio: no lens
                return torch.ops.b200vad.vad_pipeline_sincnet(r, self.packed, self.sinc, self.L, self.thr, self.kernel)
            return torch.ops.b200vad.vad_pipeline(r, lens, self.packed, self.L, self.thr, self.kernel)

        probs, decs = [], []
        for b0 in range(0, rows.shape[0], self.max_rows):
            p, d, _, _ = run(rows[b0:b0 + self.max_rows], None)
            probs.append(p); decs.append(d)
        if tail is not None:
            p, d, _, _ = run(tail, lens[-1:])
            probs.append(p); decs.append(d)
        prob = torch.cat(probs) if probs else wav.new_empty((0, Tw))
        if self.binarize is not None:
            return self._binarized(prob, N, duration, wins)
        min_run = 1 if sinc else 2      # the SincNet RLE keeps single-frame runs (predict_sincnet.py:348-370)
        if self.hop == self.window:
            # reference semantics: per-window median filter, concatenation, per-recording slice, RLE
            dec = torch.cat(decs).reshape(-1) if decs else torch.empty(0, dtype=torch.uint8, device=wav.device)
            offs = recording_offsets([duration], dec.numel(), self.fs, sincnet=sinc)
            seg, _ = torch.ops.b200vad.segments(dec, torch.tensor(offs, dtype=torch.int64, device=wav.device), min_run)
            stream = dec[: offs[1]]
        else:
            L = get_num_frames(N) if sinc else fbank_num_frames(N)       # frames of the whole recording
            sp = torch.ops.b200vad.stitch_center(prob, self.hop // (SINC_STEP if sinc else 160), L)
            stream = torch.ops.b200vad.threshold_median(sp.view(1, -1), self.thr, self.kernel, False).view(-1)
            seg, _ = torch.ops.b200vad.segments(stream.view(1, -1), None, min_run)
        ivs = segments_to_intervals(seg.tolist(), 1, self.fs, sincnet_durations=[duration] if sinc else None)[0]
        return {"prob": prob, "stream_dec": stream, "intervals": merge_intervals_with_buffer(ivs, duration, 0), "windows": wins}

    def probability_stream(self, prob: torch.Tensor, num_samples: int, duration: float) -> torch.Tensor:
        """The recording's probability stream that binarization runs over: the stitched stream for hop < window, else the
        concatenated window probabilities cut to the frames the decision stream of the reference's path covers."""
        sinc = self.sinc is not None
        if self.hop == self.window:
            flat = prob.reshape(-1)
            return flat[: recording_offsets([duration], flat.numel(), self.fs, sincnet=sinc)[1]]
        L = get_num_frames(num_samples) if sinc else fbank_num_frames(num_samples)
        return torch.ops.b200vad.stitch_center(prob, self.hop // (SINC_STEP if sinc else 160), L)

    def _binarized(self, prob, num_samples, duration, wins):
        step, t0 = mode_step(self.sinc is not None, self.fs)
        f = self.binarize.frames(step)
        sp = self.probability_stream(prob, num_samples, duration)
        dec, seg, _ = torch.ops.b200vad.binarize(sp.view(1, -1), None, f["onset"], f["offset"], f["pad_onset"], f["pad_offset"],
                                                 f["min_off"], f["min_on"])
        ivs = self.binarize.intervals(seg.tolist(), 1, step, t0, [duration])[0]
        return {"prob": prob, "stream_dec": dec.view(-1), "intervals": ivs, "windows": wins}
