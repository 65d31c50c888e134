"""torch.library custom ops over the C ABI (CUDA implementations only -- no CPU kernels).

  b200vad::fbank(wav, lens?)                        -> (B, T, 80) f32      [a1]
  b200vad::lstm_head(x, packed, num_layers)         -> (B, T) f32 prob     [a2]
  b200vad::sincnet(wav, packed)                     -> (B, Ts, 60) f32     [a3/a4]
  b200vad::threshold_median(prob, thr, kernel, i64) -> (B, T) u8 | i64     [a6/a7]
  b200vad::segments(dec, offsets?, min_run)         -> (S, 3) i32, (R) i32 [a8/a9]
  b200vad::vad_pipeline(wav, lens?, packed, L, thr, kernel) -> prob, dec, seg, counts
  b200vad::vad_pipeline_sincnet(wav, packed_model, packed_sincnet, L, thr, kernel) -> prob, dec, seg, counts
  b200vad::binarize(prob, offsets?, onset, offset, pad_onset, pad_offset, min_off, min_on) -> dec, seg, counts
  b200vad::vad_pipeline_binarize(wav, lens?, packed, packed_sincnet?, L, onset, offset, pads, min durations)
                                                    -> prob, dec, seg, counts
  b200vad::regions_step(prob, state, onset, offset, pad_onset, pad_offset, min_off, min_on, flush?)
                                                    -> ev (S, nf + 1, 2) i64, counts (S,) i32; mutates state
  b200vad::vad_pipeline_rows(wavs, rows (B, 3) host i64, window, packed, packed_sincnet?, L, thr, kernel, binarize?)
                                                    -> prob, dec, seg (padded), counts, seg_off
  b200vad::stitch_center_streams(prob, win_off, frame_off, hop_frames) -> (frame_off[-1],) f32 | u8
  b200vad::threshold_median_streams(prob, offsets, thr, kernel)       -> (n,) u8

Each op enqueues on ``torch.cuda.current_stream()`` and never synchronises, except
``segments`` / ``binarize`` and the exact-size ``vad_pipeline*`` ops, which read one int64 (the segment total) to size
their output.
"""

from __future__ import annotations

from typing import List, Optional, Tuple

import numpy as np
import torch

from . import _lib

_MAX_WS_BYTES = 40 << 30     # cap for per-call workspaces (B200: 180 GB HBM); larger batches are chunked inside the C call


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _prep(t: torch.Tensor, dtype, what: str) -> torch.Tensor:
    if not t.is_cuda:
        raise _lib.B200VadError(f"{what} must be a CUDA tensor (there is no CPU implementation of this path)")
    if t.dtype != dtype:
        raise _lib.B200VadError(f"{what} must be {dtype}, got {t.dtype}")
    return t.contiguous()


def _prep_rows(t: torch.Tensor, what: str) -> torch.Tensor:
    """(B, N) float32 (or int16 PCM) CUDA rows with unit inner stride; the row stride may be anything >= 1 (overlapping
    long-form windows are passed as an as_strided view, no copy)."""
    if not t.is_cuda:
        raise _lib.B200VadError(f"{what} must be a CUDA tensor (there is no CPU implementation of this path)")
    if t.dtype not in (torch.float32, torch.int16):
        raise _lib.B200VadError(f"{what} must be torch.float32 or torch.int16 (16-bit PCM), got {t.dtype}")
    if t.dim() == 2 and t.stride(1) == 1 and t.stride(0) >= 1:
        return t
    return t.contiguous()


def _ws(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def _ensure(device) -> int:
    idx = device.index if device.index is not None else torch.cuda.current_device()
    _lib.init(idx)
    return idx


# ------------------------------------------------------------------ fbank
@torch.library.custom_op("b200vad::fbank", mutates_args=(), device_types="cuda")
def fbank(wav: torch.Tensor, lens: Optional[torch.Tensor] = None) -> torch.Tensor:
    wav = _prep_rows(wav, "wav")
    if wav.dim() != 2:
        raise _lib.B200VadError("wav must be (B, N)")
    B, N = wav.shape
    L = _lib.lib()
    T = L.b200vad_fbank_num_frames(N)
    feats = torch.empty((B, T, 80), dtype=torch.float32, device=wav.device)
    if B == 0 or T == 0:
        return feats
    with torch.cuda.device(wav.device):
        _ensure(wav.device)
        lens_ptr = None
        if lens is not None:
            lens = _prep(lens.to(torch.int32), torch.int32, "lens")
            lens_ptr = lens.data_ptr()
        sums = torch.empty(B, dtype=torch.float64, device=wav.device)
        for b0 in range(0, B, 32768):
            b1 = min(B, b0 + 32768)
            fn = L.b200vad_fbank_i16 if wav.dtype == torch.int16 else L.b200vad_fbank_f32
            _lib.check(fn(wav.data_ptr() + wav.element_size() * b0 * wav.stride(0), None if lens_ptr is None else lens[b0:b1].data_ptr(),
                                           b1 - b0, N, wav.stride(0), feats[b0:b1].data_ptr(), T,
                                           sums[b0:b1].data_ptr(), _stream_ptr(wav.device)), "b200vad_fbank_f32")
    return feats


@fbank.register_fake
def _(wav, lens=None):
    B, N = wav.shape
    return wav.new_empty((B, (N + 80) // 160, 80), dtype=torch.float32)


# ------------------------------------------------------------------ LSTM stack + head
@torch.library.custom_op("b200vad::lstm_head", mutates_args=(), device_types="cuda")
def lstm_head(x: torch.Tensor, packed: torch.Tensor, num_layers: int) -> torch.Tensor:
    x = _prep(x, torch.float32, "x")
    if x.dim() != 3:
        raise _lib.B200VadError("x must be (B, T, D)")
    B, T, D = x.shape
    L = _lib.lib()
    if packed.numel() != L.b200vad_model_packed_bytes(D, num_layers):
        raise _lib.B200VadError("packed blob does not match (D, num_layers)")
    prob = torch.empty((B, T), dtype=torch.float32, device=x.device)
    if B == 0 or T == 0:
        return prob
    with torch.cuda.device(x.device):
        _ensure(x.device)
        need = L.b200vad_model_workspace_bytes(B, T)
        ws = _ws(min(need, max(_MAX_WS_BYTES, L.b200vad_model_workspace_bytes(1, T))), x.device)
        _lib.check(L.b200vad_model_forward_f32(packed.data_ptr(), D, num_layers, x.data_ptr(), B, T, prob.data_ptr(),
                                               ws.data_ptr(), ws.numel(), _stream_ptr(x.device)),
                   "b200vad_model_forward_f32")
    return prob


@lstm_head.register_fake
def _(x, packed, num_layers):
    return x.new_empty((x.shape[0], x.shape[1]))


# ------------------------------------------------------------------ SincNet
@torch.library.custom_op("b200vad::sincnet", mutates_args=(), device_types="cuda")
def sincnet(wav: torch.Tensor, packed: torch.Tensor) -> torch.Tensor:
    wav = _prep(wav, torch.float32, "wav")
    if wav.dim() != 2:
        raise _lib.B200VadError("wav must be (B, N)")
    B, N = wav.shape
    L = _lib.lib()
    Ts = L.b200vad_sincnet_num_frames(N)
    if Ts < 1:
        raise _lib.B200VadError("waveform shorter than the SincNet receptive field (991 samples)")
    out = torch.empty((B, Ts, 60), dtype=torch.float32, device=wav.device)
    if B == 0:
        return out
    with torch.cuda.device(wav.device):
        _ensure(wav.device)
        need = L.b200vad_sincnet_workspace_bytes(B, N)
        ws = _ws(min(need, max(_MAX_WS_BYTES, L.b200vad_sincnet_workspace_bytes(1, N))), wav.device)
        _lib.check(L.b200vad_sincnet_forward_f32(packed.data_ptr(), wav.data_ptr(), B, N, wav.stride(0), out.data_ptr(),
                                                 ws.data_ptr(), ws.numel(), _stream_ptr(wav.device)),
                   "b200vad_sincnet_forward_f32")
    return out


@sincnet.register_fake
def _(wav, packed):
    from .host import get_num_frames
    return wav.new_empty((wav.shape[0], get_num_frames(wav.shape[1]), 60))


# ------------------------------------------------------------------ threshold + median
@torch.library.custom_op("b200vad::threshold_median", mutates_args=(), device_types="cuda")
def threshold_median(prob: torch.Tensor, thr: float, kernel: int, as_int64: bool) -> torch.Tensor:
    prob = _prep(prob, torch.float32, "prob")
    if prob.dim() != 2:
        raise _lib.B200VadError("prob must be (B, T)")
    B, T = prob.shape
    out = torch.empty((B, T), dtype=torch.int64 if as_int64 else torch.uint8, device=prob.device)
    if B == 0 or T == 0:
        return out
    L = _lib.lib()
    with torch.cuda.device(prob.device):
        for b0 in range(0, B, 32768):
            b1 = min(B, b0 + 32768)
            _lib.check(L.b200vad_threshold_median(prob[b0:b1].data_ptr(), b1 - b0, T, float(thr), int(kernel),
                                                  out[b0:b1].data_ptr(), 8 if as_int64 else 1, None, 0.0,
                                                  _stream_ptr(prob.device)), "b200vad_threshold_median")
    return out


@threshold_median.register_fake
def _(prob, thr, kernel, as_int64):
    return prob.new_empty(prob.shape, dtype=torch.int64 if as_int64 else torch.uint8)


def near_threshold_count(prob: torch.Tensor, thr: float, tol: float) -> int:
    """Number of frames with |p - thr| <= tol (reported separately by the parity tests)."""
    return int(((prob - thr).abs() <= tol).sum().item())


# ------------------------------------------------------------------ segments
@torch.library.custom_op("b200vad::segments", mutates_args=(), device_types="cuda")
def segments(dec: torch.Tensor, offsets: Optional[torch.Tensor] = None, min_run: int = 2) -> Tuple[torch.Tensor, torch.Tensor]:
    dec = _prep(dec, torch.uint8, "dec")
    L = _lib.lib()
    dev = dec.device
    if offsets is None:
        if dec.dim() != 2:
            raise _lib.B200VadError("dec must be (R, T) when offsets is None")
        R, T = dec.shape
        total_frames = R * T
        off_ptr = None
    else:
        offsets = _prep(offsets.to(torch.int64), torch.int64, "offsets")
        R, T = offsets.numel() - 1, 0
        total_frames = dec.numel()
        off_ptr = offsets.data_ptr()
    counts = torch.zeros(max(R, 0), dtype=torch.int32, device=dev)
    if R <= 0:
        return torch.empty((0, 3), dtype=torch.int32, device=dev), counts
    cap = total_frames // max(min_run + 1, 2) + R + 1
    seg_off = torch.empty(R + 1, dtype=torch.int64, device=dev)
    seg = torch.empty((cap, 3), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.b200vad_segments(dec.data_ptr(), off_ptr, R, T, int(min_run), counts.data_ptr(), seg_off.data_ptr(),
                                      seg.data_ptr(), cap, _stream_ptr(dev)), "b200vad_segments")
    total = int(seg_off[R].item())
    return seg[:total].clone(), counts


@segments.register_fake
def _(dec, offsets=None, min_run=2):
    ctx = torch.library.get_ctx()
    n = ctx.new_dynamic_size()
    R = dec.shape[0] if offsets is None else offsets.numel() - 1
    return dec.new_empty((n, 3), dtype=torch.int32), dec.new_empty((R,), dtype=torch.int32)


# ------------------------------------------------------------------ binarization (onset / offset hysteresis, pads, min durations)
def _bin_params(onset, offset, pad_onset, pad_offset, min_off, min_on):
    return _lib.BinarizeParams(float(onset), float(offset), int(pad_onset), int(pad_offset), int(min_off), int(min_on))


@torch.library.custom_op("b200vad::binarize", mutates_args=(), device_types="cuda")
def binarize(prob: torch.Tensor, offsets: Optional[torch.Tensor], onset: float, offset: float, pad_onset: int, pad_offset: int,
             min_off: int, min_on: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """pyannote's Binarize in frames (include/b200vad.h): prob (R, T) rows, or a flat (n,) buffer with offsets (R+1) int64 ->
    dec (same shape) uint8, seg (S, 3) int32 (stream, first, last) ordered by (stream, first), counts (R,) int32.  One blocking
    read of the region total to size seg.  b200vad.Binarize converts a policy in seconds to these frame counts."""
    prob = _prep(prob, torch.float32, "prob")
    dev = prob.device
    if offsets is None:
        if prob.dim() != 2:
            raise _lib.B200VadError("prob must be (R, T) when offsets is None")
        R, T = prob.shape
        cap = R * ((T + 1) // 2)
        off_ptr = None
    else:
        if prob.dim() != 1:
            raise _lib.B200VadError("prob must be a flat (n,) buffer when offsets are given")
        offsets = _prep(offsets.to(torch.int64), torch.int64, "offsets")
        R, T = offsets.numel() - 1, prob.numel()
        cap = (T + R) // 2 + 1          # >= sum of ceil(len_r / 2) over R streams of at most T frames in all
        off_ptr = offsets.data_ptr()
    dec = torch.empty(prob.shape, dtype=torch.uint8, device=dev)
    counts = torch.zeros(max(R, 0), dtype=torch.int32, device=dev)
    if R <= 0:
        return dec.zero_(), torch.empty((0, 3), dtype=torch.int32, device=dev), counts
    seg_off = torch.empty(R + 1, dtype=torch.int64, device=dev)
    seg = torch.empty((cap, 3), dtype=torch.int32, device=dev)
    params = _bin_params(onset, offset, pad_onset, pad_offset, min_off, min_on)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().b200vad_binarize(prob.data_ptr(), off_ptr, R, T, params, dec.data_ptr(), counts.data_ptr(),
                                               seg_off.data_ptr(), seg.data_ptr(), cap, _stream_ptr(dev)), "b200vad_binarize")
    total = int(seg_off[R].item())
    return dec, seg[:total].clone(), counts


@binarize.register_fake
def _(prob, offsets, onset, offset, pad_onset, pad_offset, min_off, min_on):
    ctx = torch.library.get_ctx()
    n = ctx.new_dynamic_size()
    R = prob.shape[0] if offsets is None else offsets.numel() - 1
    return prob.new_empty(prob.shape, dtype=torch.uint8), prob.new_empty((n, 3), dtype=torch.int32), prob.new_empty((R,), dtype=torch.int32)


@torch.library.custom_op("b200vad::regions_step", mutates_args=("state",), device_types="cuda")
def regions_step(prob: torch.Tensor, state: torch.Tensor, onset: float, offset: float, pad_onset: int, pad_offset: int, min_off: int,
                 min_on: int, flush: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Speech start / end events on streams fed a chunk at a time (include/b200vad.h, b200vad_regions_step): prob (S, nf) f32
    are the next nf frames of S streams, state (S, 5) int64 (zeros = fresh streams) is advanced in place.  Returns ev
    (S, nf + 1, 2) int64 rows (frame, kind: 1 start / 0 end), of which the first counts[r] of stream r are valid (the rest
    unspecified), and counts (S,) int32.  flush (S,) bool, optional: those streams end after their frames (their open group is
    closed, their state zeroed).  Never synchronises."""
    prob = _prep(prob, torch.float32, "prob")
    if prob.dim() != 2:
        raise _lib.B200VadError("prob must be (S, nf)")
    S, nf = prob.shape
    if state.dtype != torch.int64 or tuple(state.shape) != (S, 5) or not state.is_contiguous() or state.device != prob.device:
        raise _lib.B200VadError("state must be a contiguous (S, 5) int64 tensor on prob's device")
    dev = prob.device
    flush_ptr = None
    if flush is not None:
        if flush.numel() != S:
            raise _lib.B200VadError("flush must hold one flag per stream")
        flush = _prep(flush.reshape(S).to(torch.uint8), torch.uint8, "flush")
        flush_ptr = flush.data_ptr()
    ev = torch.empty((S, nf + 1, 2), dtype=torch.int64, device=dev)
    counts = torch.empty(S, dtype=torch.int32, device=dev)
    params = _bin_params(onset, offset, pad_onset, pad_offset, min_off, min_on)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().b200vad_regions_step(prob.data_ptr() if prob.numel() else None, S, nf, nf, params, state.data_ptr(),
                                                   flush_ptr, ev.data_ptr(), counts.data_ptr(), nf + 1, _stream_ptr(dev)),
                   "b200vad_regions_step")
    return ev, counts


@regions_step.register_fake
def _(prob, state, onset, offset, pad_onset, pad_offset, min_off, min_on, flush=None):
    S, nf = prob.shape
    return prob.new_empty((S, nf + 1, 2), dtype=torch.int64), prob.new_empty((S,), dtype=torch.int32)


# ------------------------------------------------------------------ whole path
def _seg_per_row(T: int, sincnet: bool) -> int:
    """Most segments a row of T frames can hold: runs of >= 2 frames (fbank path) or of >= 1 frame (the SincNet RLE,
    predict_sincnet.py:348-370)."""
    return (T + 1) // 2 if sincnet else (T + 2) // 3


def _pipeline_launch(wav, lens, packed, num_layers, thr, kernel, sinc=None, bin=None):
    """Enqueues the whole path on the current stream; returns device buffers only (nothing synchronises):
    prob (B, T) f32, dec (B, T) u8, seg (cap, 3) i32 of which the first seg_off[B] rows are valid, counts (B,) i32,
    seg_off (B + 1,) i64.  ``sinc``: packed SincNet blob -> the SincNet -> PyanNet path (then ``lens`` must be None).
    ``bin``: BinarizeParams -> binarization instead of threshold / median / segments (thr and kernel unused; the segment
    capacity is B * ceil(T / 2))."""
    wav = _prep_rows(wav, "wav")
    if wav.dim() != 2:
        raise _lib.B200VadError("wav must be (B, N)")
    B, N = wav.shape
    L = _lib.lib()
    dev = wav.device
    if sinc is None:
        T = L.b200vad_fbank_num_frames(N)
    else:
        T = L.b200vad_sincnet_num_frames(N)
        if T < 1:
            raise _lib.B200VadError("waveform shorter than the SincNet receptive field (991 samples)")
    prob = torch.empty((B, T), dtype=torch.float32, device=dev)
    dec = torch.empty((B, T), dtype=torch.uint8, device=dev)
    counts = torch.zeros(B, dtype=torch.int32, device=dev)
    seg_off = torch.zeros(B + 1, dtype=torch.int64, device=dev)
    if B == 0 or T == 0:
        return prob, dec, torch.empty((0, 3), dtype=torch.int32, device=dev), counts, seg_off
    if B > _MAX_PIPELINE_ROWS:
        raise _lib.B200VadError(f"one pipeline launch handles at most {_MAX_PIPELINE_ROWS} rows (vad_pipeline splits larger batches)")
    cap = B * ((T + 1) // 2 if bin is not None else _seg_per_row(T, sinc is not None))
    seg = torch.empty((cap, 3), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _ensure(dev)
        lens_ptr = None
        if lens is not None:
            lens = _prep(lens.to(torch.int32), torch.int32, "lens")
            lens_ptr = lens.data_ptr()
        ws = _pipeline_ws(B, N, T, sinc is not None, dev)
        if sinc is None:
            if bin is not None:
                _lib.check(L.b200vad_pipeline_binarize(packed.data_ptr(), None, num_layers, wav.data_ptr(), int(wav.dtype == torch.int16),
                                                       lens_ptr, B, N, wav.stride(0), bin, prob.data_ptr(), dec.data_ptr(),
                                                       counts.data_ptr(), seg_off.data_ptr(), seg.data_ptr(), cap, ws.data_ptr(),
                                                       ws.numel(), _stream_ptr(dev)), "b200vad_pipeline_binarize")
                return prob, dec, seg, counts, seg_off
            fn = L.b200vad_pipeline_fbank_i16 if wav.dtype == torch.int16 else L.b200vad_pipeline_fbank_f32
            _lib.check(fn(packed.data_ptr(), num_layers, wav.data_ptr(), lens_ptr, B, N, wav.stride(0),
                          float(thr), int(kernel), prob.data_ptr(), dec.data_ptr(), counts.data_ptr(),
                          seg_off.data_ptr(), seg.data_ptr(), cap, ws.data_ptr(), ws.numel(),
                          _stream_ptr(dev)), "b200vad_pipeline_fbank_f32")
        else:
            if lens is not None:
                raise _lib.B200VadError("the SincNet path takes no lens: pad rows with zero audio, as the reference does")
            if bin is not None:
                _lib.check(L.b200vad_pipeline_binarize(packed.data_ptr(), sinc.data_ptr(), num_layers, wav.data_ptr(),
                                                       int(wav.dtype == torch.int16), None, B, N, wav.stride(0), bin, prob.data_ptr(),
                                                       dec.data_ptr(), counts.data_ptr(), seg_off.data_ptr(), seg.data_ptr(), cap,
                                                       ws.data_ptr(), ws.numel(), _stream_ptr(dev)), "b200vad_pipeline_binarize")
                return prob, dec, seg, counts, seg_off
            fn = L.b200vad_pipeline_sincnet_i16 if wav.dtype == torch.int16 else L.b200vad_pipeline_sincnet_f32
            _lib.check(fn(packed.data_ptr(), sinc.data_ptr(), num_layers, wav.data_ptr(), B, N, wav.stride(0),
                          float(thr), int(kernel), prob.data_ptr(), dec.data_ptr(), counts.data_ptr(),
                          seg_off.data_ptr(), seg.data_ptr(), cap, ws.data_ptr(), ws.numel(),
                          _stream_ptr(dev)), "b200vad_pipeline_sincnet_f32")
    return prob, dec, seg, counts, seg_off


_MAX_PIPELINE_ROWS = 65535        # grid limit of the per-row kernels behind one C call


def _pipeline_ws(B: int, N: int, T: int, sincnet: bool, dev) -> torch.Tensor:
    """Workspace of one pipeline launch of B rows of N samples (T frames), capped at _MAX_WS_BYTES unless the launch needs more."""
    L = _lib.lib()
    if not sincnet:
        need = L.b200vad_pipeline_workspace_bytes(B, N)
        minimum = need - L.b200vad_model_workspace_bytes(B, T) + L.b200vad_model_workspace_bytes(1, T)
    else:
        need = L.b200vad_pipeline_sincnet_workspace_bytes(B, N)
        minimum = 256 * B * T + L.b200vad_pipeline_sincnet_workspace_bytes(1, N)    # + the whole batch's layer-0 planes
    return _ws(min(need, max(_MAX_WS_BYTES, minimum)), dev)


def _upload(values, dtype, dev) -> torch.Tensor:
    """Host list or array -> device tensor through pinned memory: enqueued on the current stream, no synchronisation."""
    return torch.as_tensor(np.asarray(values)).to(dtype).pin_memory().to(dev, non_blocking=True)


# ------------------------------------------------------------------ windows of many recordings: rows through a pointer table
@torch.library.custom_op("b200vad::vad_pipeline_rows", mutates_args=(), device_types="cuda")
def vad_pipeline_rows(wavs: List[torch.Tensor], rows: torch.Tensor, window: int, packed: torch.Tensor,
                      packed_sincnet: Optional[torch.Tensor], num_layers: int, thr: float, kernel: int,
                      binarize: Optional[List[float]] = None
                      ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """The whole path on B rows of ``window`` samples cut from several recordings (b200vad_pipeline_rows): ``rows`` is a (B, 3)
    int64 host tensor of (recording, start, valid), and row b reads wavs[recording][start : start + valid] only, in place.
    wavs: contiguous 1-D CUDA tensors on one device, all float32 or all int16 PCM.  fbank (packed_sincnet None): features past
    the valid frames are LOG_EPS, as lens means for vad_pipeline; SincNet: samples past the valid ones are zeros.
    ``binarize``: [onset, offset, pad_onset, pad_offset, min_off, min_on] -> binarization instead of threshold / median.
    Returns what vad_pipeline_padded does -- prob (B, T), dec (B, T), seg at its fixed capacity, counts (B,), seg_off (B + 1,)
    -- without any host synchronisation; the recordings must stay alive until the work on the current stream is done."""
    if not wavs:
        raise _lib.B200VadError("wavs is empty")
    dev, dtype = wavs[0].device, wavs[0].dtype
    if dtype not in (torch.float32, torch.int16):
        raise _lib.B200VadError(f"wavs must be torch.float32 or torch.int16 (16-bit PCM), got {dtype}")
    for i, w in enumerate(wavs):
        if not w.is_cuda or w.device != dev or w.dtype != dtype or w.dim() != 1 or not w.is_contiguous():
            raise _lib.B200VadError(f"wavs[{i}] must be a contiguous 1-D {dtype} tensor on {dev}")
    if rows.device.type != "cpu" or rows.dim() != 2 or rows.shape[1] != 3:
        raise _lib.B200VadError("rows must be a (B, 3) host tensor of (recording, start, valid)")
    B, N = rows.shape[0], int(window)
    L = _lib.lib()
    sinc = packed_sincnet is not None
    T = L.b200vad_sincnet_num_frames(N) if sinc else L.b200vad_fbank_num_frames(N)
    if sinc and T < 1:
        raise _lib.B200VadError("window shorter than the SincNet receptive field (991 samples)")
    if B > _MAX_PIPELINE_ROWS:
        raise _lib.B200VadError(f"one pipeline launch handles at most {_MAX_PIPELINE_ROWS} rows")
    tab = rows.to(torch.int64).numpy()
    rec, start, valid = tab[:, 0], tab[:, 1], tab[:, 2]
    numel = np.asarray([w.numel() for w in wavs], dtype=np.int64)
    ok = (rec >= 0) & (rec < len(wavs)) & (start >= 0) & (valid >= 0) & (valid <= N)
    ok[ok] &= start[ok] + valid[ok] <= numel[rec[ok]]
    if not ok.all():
        b = int(np.flatnonzero(~ok)[0])
        raise _lib.B200VadError(f"row {b}: {tuple(tab[b].tolist())} is not inside a recording or longer than the window")
    # one upload: B row pointers, then the B int32 valid lengths packed two to an int64 word
    base = np.asarray([w.data_ptr() for w in wavs], dtype=np.int64)
    table = np.zeros(B + (B + 1) // 2, dtype=np.int64)
    table[:B] = base[rec] + wavs[0].element_size() * start
    table[B:].view(np.int32)[:B] = valid
    prob = torch.empty((B, T), dtype=torch.float32, device=dev)
    dec = torch.empty((B, T), dtype=torch.uint8, device=dev)
    counts = torch.zeros(B, dtype=torch.int32, device=dev)
    seg_off = torch.zeros(B + 1, dtype=torch.int64, device=dev)
    if B == 0 or T == 0:
        return prob, dec, torch.empty((0, 3), dtype=torch.int32, device=dev), counts, seg_off
    bin = _bin_params(*binarize) if binarize is not None else None
    cap = B * ((T + 1) // 2 if bin is not None else _seg_per_row(T, sinc))
    seg = torch.empty((cap, 3), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _ensure(dev)
        table_d = _upload(table, torch.int64, dev)
        ws = _pipeline_ws(B, N, T, sinc, dev)
        _lib.check(L.b200vad_pipeline_rows(packed.data_ptr(), packed_sincnet.data_ptr() if sinc else None, num_layers, table_d.data_ptr(),
                                           int(dtype == torch.int16), table_d.data_ptr() + 8 * B, B, N, float(thr), int(kernel), bin,
                                           prob.data_ptr(), dec.data_ptr(), counts.data_ptr(), seg_off.data_ptr(), seg.data_ptr(), cap,
                                           ws.data_ptr(), ws.numel(), _stream_ptr(dev)), "b200vad_pipeline_rows")
    return prob, dec, seg, counts, seg_off


@vad_pipeline_rows.register_fake
def _(wavs, rows, window, packed, packed_sincnet, num_layers, thr, kernel, binarize=None):
    B, N = rows.shape[0], int(window)
    T = (N + 80) // 160 if packed_sincnet is None else _sincnet_frames(N)
    cap = B * ((T + 1) // 2 if binarize is not None else _seg_per_row(T, packed_sincnet is not None))
    w = wavs[0]
    return (w.new_empty((B, T), dtype=torch.float32), w.new_empty((B, T), dtype=torch.uint8), w.new_empty((cap, 3), dtype=torch.int32),
            w.new_empty((B,), dtype=torch.int32), w.new_empty((B + 1,), dtype=torch.int64))


@torch.library.custom_op("b200vad::vad_pipeline_padded", mutates_args=(), device_types="cuda")
def vad_pipeline_padded(wav: torch.Tensor, lens: Optional[torch.Tensor], packed: torch.Tensor, num_layers: int, thr: float,
                        kernel: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """The whole path without any host synchronisation: the segment list comes back at its fixed capacity
    (B * ceil(T / 3) rows) together with the per-row offsets; rows [0, seg_off[B]) are valid.  For pipelines that keep the
    stream full (bench.py, b200vad.SegmentGatherer)."""
    return _pipeline_launch(wav, lens, packed, num_layers, thr, kernel)


@vad_pipeline_padded.register_fake
def _(wav, lens, packed, num_layers, thr, kernel):
    B, N = wav.shape
    T = (N + 80) // 160
    return (wav.new_empty((B, T), dtype=torch.float32), wav.new_empty((B, T), dtype=torch.uint8),
            wav.new_empty((B * ((T + 2) // 3), 3), dtype=torch.int32), wav.new_empty((B,), dtype=torch.int32),
            wav.new_empty((B + 1,), dtype=torch.int64))


@torch.library.custom_op("b200vad::vad_pipeline", mutates_args=(), device_types="cuda")
def vad_pipeline(wav: torch.Tensor, lens: Optional[torch.Tensor], packed: torch.Tensor, num_layers: int, thr: float,
                 kernel: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """prob, dec, seg (S, 3), counts.  The exact-size segment list needs S on the host: ONE blocking read of the total per
    call, after everything is enqueued (use vad_pipeline_padded to avoid it).  Batches of more than 65 535 rows are split."""
    return _pipeline_exact(wav, lens, packed, num_layers, thr, kernel)


def _pipeline_exact(wav, lens, packed, num_layers, thr, kernel, sinc=None, bin=None):
    B = wav.shape[0]
    if B <= _MAX_PIPELINE_ROWS:
        prob, dec, seg, counts, seg_off = _pipeline_launch(wav, lens, packed, num_layers, thr, kernel, sinc, bin)
        total = int(seg_off[B].item()) if B > 0 else 0
        return prob, dec, seg[:total].clone(), counts
    outs = []
    for b0 in range(0, B, _MAX_PIPELINE_ROWS):
        sl = slice(b0, min(B, b0 + _MAX_PIPELINE_ROWS))
        outs.append((b0,) + _pipeline_launch(wav[sl], None if lens is None else lens[sl], packed, num_layers, thr, kernel, sinc,
                                             bin))
    segs = []
    for b0, _, _, seg, _, seg_off in outs:
        s = seg[: int(seg_off[-1].item())].clone()
        s[:, 0] += b0
        segs.append(s)
    return (torch.cat([o[1] for o in outs]), torch.cat([o[2] for o in outs]), torch.cat(segs), torch.cat([o[4] for o in outs]))


@vad_pipeline.register_fake
def _(wav, lens, packed, num_layers, thr, kernel):
    ctx = torch.library.get_ctx()
    n = ctx.new_dynamic_size()
    B, N = wav.shape
    T = (N + 80) // 160
    return (wav.new_empty((B, T), dtype=torch.float32), wav.new_empty((B, T), dtype=torch.uint8), wav.new_empty((n, 3), dtype=torch.int32),
            wav.new_empty((B,), dtype=torch.int32))


def _sincnet_frames(N: int) -> int:
    from .host import get_num_frames
    return get_num_frames(N)


@torch.library.custom_op("b200vad::vad_pipeline_sincnet_padded", mutates_args=(), device_types="cuda")
def vad_pipeline_sincnet_padded(wav: torch.Tensor, packed_model: torch.Tensor, packed_sincnet: torch.Tensor, num_layers: int,
                                thr: float, kernel: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """vad_pipeline_padded on the SincNet -> PyanNet path (the reference's feature_extractor="sincnet" flow): prob / dec
    (B, Ts), Ts = get_num_frames(N); segments keep single-frame runs (predict_sincnet.py:348-370), so the fixed capacity is
    B * ceil(Ts / 2) rows.  wav: (B, N) float32 or int16 PCM rows, N >= 991; pad short audio with zeros (no lens)."""
    return _pipeline_launch(wav, None, packed_model, num_layers, thr, kernel, packed_sincnet)


@vad_pipeline_sincnet_padded.register_fake
def _(wav, packed_model, packed_sincnet, num_layers, thr, kernel):
    B, N = wav.shape
    T = _sincnet_frames(N)
    return (wav.new_empty((B, T), dtype=torch.float32), wav.new_empty((B, T), dtype=torch.uint8),
            wav.new_empty((B * _seg_per_row(T, True), 3), dtype=torch.int32), wav.new_empty((B,), dtype=torch.int32),
            wav.new_empty((B + 1,), dtype=torch.int64))


@torch.library.custom_op("b200vad::vad_pipeline_sincnet", mutates_args=(), device_types="cuda")
def vad_pipeline_sincnet(wav: torch.Tensor, packed_model: torch.Tensor, packed_sincnet: torch.Tensor, num_layers: int, thr: float,
                         kernel: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """vad_pipeline on the SincNet -> PyanNet path: prob (B, Ts), dec (B, Ts), seg (S, 3) with single-frame runs kept (min_run
    1), counts.  One blocking read of the segment total per call; batches of more than 65 535 rows are split."""
    return _pipeline_exact(wav, None, packed_model, num_layers, thr, kernel, packed_sincnet)


@vad_pipeline_sincnet.register_fake
def _(wav, packed_model, packed_sincnet, num_layers, thr, kernel):
    ctx = torch.library.get_ctx()
    n = ctx.new_dynamic_size()
    B, N = wav.shape
    T = _sincnet_frames(N)
    return (wav.new_empty((B, T), dtype=torch.float32), wav.new_empty((B, T), dtype=torch.uint8), wav.new_empty((n, 3), dtype=torch.int32),
            wav.new_empty((B,), dtype=torch.int32))


def _pipeline_frames(wav, packed_sincnet) -> int:
    N = wav.shape[1]
    return (N + 80) // 160 if packed_sincnet is None else _sincnet_frames(N)


@torch.library.custom_op("b200vad::vad_pipeline_binarize_padded", mutates_args=(), device_types="cuda")
def vad_pipeline_binarize_padded(wav: torch.Tensor, lens: Optional[torch.Tensor], packed: torch.Tensor,
                                 packed_sincnet: Optional[torch.Tensor], num_layers: int, onset: float, offset: float, pad_onset: int,
                                 pad_offset: int, min_off: int, min_on: int
                                 ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """The whole path with binarization (``binarize`` on prob) and no host synchronisation: the fbank front end, or SincNet with
    ``packed_sincnet`` (then ``lens`` must be None); float32 or int16 PCM rows.  prob equals vad_pipeline / vad_pipeline_sincnet
    bit for bit.  The segment list comes back at its fixed capacity B * ceil(T / 2) with seg_off (B + 1,); rows [0, seg_off[B])
    are valid (b200vad.SegmentGatherer takes them as they are)."""
    return _pipeline_launch(wav, lens, packed, num_layers, 0.5, 49, packed_sincnet,
                            _bin_params(onset, offset, pad_onset, pad_offset, min_off, min_on))


@vad_pipeline_binarize_padded.register_fake
def _(wav, lens, packed, packed_sincnet, num_layers, onset, offset, pad_onset, pad_offset, min_off, min_on):
    B = wav.shape[0]
    T = _pipeline_frames(wav, packed_sincnet)
    return (wav.new_empty((B, T), dtype=torch.float32), wav.new_empty((B, T), dtype=torch.uint8),
            wav.new_empty((B * ((T + 1) // 2), 3), dtype=torch.int32), wav.new_empty((B,), dtype=torch.int32),
            wav.new_empty((B + 1,), dtype=torch.int64))


@torch.library.custom_op("b200vad::vad_pipeline_binarize", mutates_args=(), device_types="cuda")
def vad_pipeline_binarize(wav: torch.Tensor, lens: Optional[torch.Tensor], packed: torch.Tensor, packed_sincnet: Optional[torch.Tensor],
                          num_layers: int, onset: float, offset: float, pad_onset: int, pad_offset: int, min_off: int,
                          min_on: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """vad_pipeline_binarize_padded with an exact-size segment list: prob, dec, seg (S, 3), counts.  One blocking read of the
    segment total per call; batches of more than 65 535 rows are split."""
    return _pipeline_exact(wav, lens, packed, num_layers, 0.5, 49, packed_sincnet,
                           _bin_params(onset, offset, pad_onset, pad_offset, min_off, min_on))


@vad_pipeline_binarize.register_fake
def _(wav, lens, packed, packed_sincnet, num_layers, onset, offset, pad_onset, pad_offset, min_off, min_on):
    ctx = torch.library.get_ctx()
    n = ctx.new_dynamic_size()
    B = wav.shape[0]
    T = _pipeline_frames(wav, packed_sincnet)
    return (wav.new_empty((B, T), dtype=torch.float32), wav.new_empty((B, T), dtype=torch.uint8), wav.new_empty((n, 3), dtype=torch.int32),
            wav.new_empty((B,), dtype=torch.int32))


# ------------------------------------------------------------------ scoring (SURVEY 8f rank 1)
@torch.library.custom_op("b200vad::stat_scores", mutates_args=(), device_types="cuda")
def stat_scores(dec: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
    """(tp, fp, tn, fn) int64 of decisions (uint8, != 0 is speech) against labels (uint8)."""
    dec = _prep(dec, torch.uint8, "dec").reshape(-1)
    labels = _prep(labels, torch.uint8, "labels").reshape(-1)
    if dec.numel() != labels.numel():
        raise _lib.B200VadError("dec and labels must have the same number of frames")
    out = torch.empty(4, dtype=torch.int64, device=dec.device)
    with torch.cuda.device(dec.device):
        _lib.check(_lib.lib().b200vad_stat_scores(dec.data_ptr(), labels.data_ptr(), dec.numel(), out.data_ptr(),
                                                  _stream_ptr(dec.device)), "b200vad_stat_scores")
    return out


@stat_scores.register_fake
def _(dec, labels):
    return dec.new_empty((4,), dtype=torch.int64)


@torch.library.custom_op("b200vad::score_intervals", mutates_args=(), device_types="cuda")
def score_intervals(gt_iv: torch.Tensor, pred_iv: torch.Tensor, word_off: torch.Tensor, nframes: torch.Tensor,
                    total_words: int, max_words_per_rec: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """gt_iv / pred_iv: (n, 3) int32 (recording, start_frame, end_frame_exclusive); word_off (R+1) int64;
    nframes (R) int32 -> per-recording false-alarm and missed frame counts (R) int64."""
    gt_iv = _prep(gt_iv, torch.int32, "gt_iv")
    pred_iv = _prep(pred_iv, torch.int32, "pred_iv")
    word_off = _prep(word_off, torch.int64, "word_off")
    nframes = _prep(nframes, torch.int32, "nframes")
    dev = nframes.device
    R = nframes.numel()
    fa = torch.zeros(R, dtype=torch.int64, device=dev)
    md = torch.zeros(R, dtype=torch.int64, device=dev)
    if R == 0:
        return fa, md
    L = _lib.lib()
    ws = _ws(L.b200vad_score_workspace_bytes(total_words), dev)
    with torch.cuda.device(dev):
        _lib.check(L.b200vad_score_intervals(gt_iv.data_ptr() if gt_iv.numel() else None, gt_iv.shape[0],
                                             pred_iv.data_ptr() if pred_iv.numel() else None, pred_iv.shape[0],
                                             word_off.data_ptr(), nframes.data_ptr(), R, int(total_words), int(max_words_per_rec),
                                             ws.data_ptr(), fa.data_ptr(), md.data_ptr(), _stream_ptr(dev)),
                   "b200vad_score_intervals")
    return fa, md


@score_intervals.register_fake
def _(gt_iv, pred_iv, word_off, nframes, total_words, max_words_per_rec):
    R = nframes.shape[0]
    return nframes.new_empty((R,), dtype=torch.int64), nframes.new_empty((R,), dtype=torch.int64)


# ------------------------------------------------------------------ long-form stitching (BASELINE config 3)
@torch.library.custom_op("b200vad::stitch_center", mutates_args=(), device_types="cuda")
def stitch_center(prob: torch.Tensor, hop_frames: int, total_frames: int) -> torch.Tensor:
    """prob (W, Tw) of windows starting every hop_frames frames -> stitched (total_frames,) stream."""
    prob = _prep(prob, torch.float32, "prob")
    if prob.dim() != 2:
        raise _lib.B200VadError("prob must be (W, Tw)")
    W, Tw = prob.shape
    out = torch.empty(int(total_frames), dtype=torch.float32, device=prob.device)
    with torch.cuda.device(prob.device):
        _lib.check(_lib.lib().b200vad_stitch_center(prob.data_ptr(), W, Tw, int(hop_frames), out.data_ptr(), int(total_frames),
                                                    _stream_ptr(prob.device)), "b200vad_stitch_center")
    return out


@stitch_center.register_fake
def _(prob, hop_frames, total_frames):
    return prob.new_empty((total_frames,))


def _check_offsets(off: List[int], end: int, what: str) -> None:
    if len(off) < 1 or off[0] != 0 or off[-1] != end or any(b < a for a, b in zip(off, off[1:])):
        raise _lib.B200VadError(f"{what} must rise from 0 to {end}")


_MAX_STREAMS = 65535              # grid limit of the ragged kernels behind one C call


@torch.library.custom_op("b200vad::stitch_center_streams", mutates_args=(), device_types="cuda")
def stitch_center_streams(prob: torch.Tensor, win_off: List[int], frame_off: List[int], hop_frames: int) -> torch.Tensor:
    """stitch_center for R recordings at once (b200vad_stitch_center_streams): prob (W, Tw) float32 probabilities or uint8
    decisions; recording r has the windows prob[win_off[r] : win_off[r + 1]] and its stitched stream is
    out[frame_off[r] : frame_off[r + 1]] (host lists of R + 1 offsets from 0).  Frames no window covers are 0.  With
    hop_frames = Tw each stream is its windows concatenated and cut to its length.  More than 65 535 recordings are split
    across launches."""
    if not prob.is_cuda or prob.dtype not in (torch.float32, torch.uint8) or prob.dim() != 2:
        raise _lib.B200VadError("prob must be a (W, Tw) float32 or uint8 CUDA tensor")
    prob = prob.contiguous()
    W, Tw = prob.shape
    R = len(win_off) - 1
    if len(frame_off) != R + 1:
        raise _lib.B200VadError("win_off and frame_off must both hold R + 1 offsets")
    _check_offsets(win_off, W, "win_off")
    _check_offsets(frame_off, frame_off[-1] if frame_off else 0, "frame_off")
    dev = prob.device
    out = torch.empty(frame_off[-1], dtype=prob.dtype, device=dev)
    if out.numel() == 0:
        return out
    with torch.cuda.device(dev):
        off = _upload(win_off + frame_off, torch.int64, dev)
        wo, fo = off[:R + 1], off[R + 1:]
        for r0 in range(0, R, _MAX_STREAMS):
            r1 = min(R, r0 + _MAX_STREAMS)
            max_len = max(b - a for a, b in zip(frame_off[r0:r1], frame_off[r0 + 1:r1 + 1]))
            _lib.check(_lib.lib().b200vad_stitch_center_streams(prob.data_ptr(), prob.element_size(), wo[r0:].data_ptr(), fo[r0:].data_ptr(),
                                                                r1 - r0, Tw, int(hop_frames), max_len, out.data_ptr(),
                                                                _stream_ptr(dev)), "b200vad_stitch_center_streams")
    return out


@stitch_center_streams.register_fake
def _(prob, win_off, frame_off, hop_frames):
    return prob.new_empty((frame_off[-1],))


@torch.library.custom_op("b200vad::threshold_median_streams", mutates_args=(), device_types="cuda")
def threshold_median_streams(prob: torch.Tensor, offsets: List[int], thr: float, kernel: int) -> torch.Tensor:
    """threshold_median on R ragged streams of a flat (n,) float32 buffer (b200vad_threshold_median_streams): stream r is
    prob[offsets[r] : offsets[r + 1]] (host list of R + 1 offsets from 0 to n), zero padded at its own edges.  Returns (n,)
    uint8.  More than 65 535 streams are split across launches."""
    prob = _prep(prob, torch.float32, "prob")
    if prob.dim() != 1:
        raise _lib.B200VadError("prob must be a flat (n,) buffer")
    _check_offsets(offsets, prob.numel(), "offsets")
    dev = prob.device
    out = torch.empty(prob.numel(), dtype=torch.uint8, device=dev)
    if out.numel() == 0:
        return out
    R = len(offsets) - 1
    with torch.cuda.device(dev):
        off = _upload(offsets, torch.int64, dev)
        for r0 in range(0, R, _MAX_STREAMS):
            r1 = min(R, r0 + _MAX_STREAMS)
            max_len = max(b - a for a, b in zip(offsets[r0:r1], offsets[r0 + 1:r1 + 1]))
            _lib.check(_lib.lib().b200vad_threshold_median_streams(prob.data_ptr(), off[r0:].data_ptr(), r1 - r0, max_len, float(thr),
                                                                   int(kernel), out.data_ptr(), _stream_ptr(dev)),
                       "b200vad_threshold_median_streams")
    return out


@threshold_median_streams.register_fake
def _(prob, offsets, thr, kernel):
    return prob.new_empty(prob.shape, dtype=torch.uint8)
