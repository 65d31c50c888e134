"""Streaming mode (BASELINE config 5): many concurrent streams, small hops, per-chunk latency.

No reference semantics exist (the BiLSTM is non-causal, DC removal is whole-signal), so the mode is defined as
(SURVEY 8a "streaming"): every stream keeps the last ``window`` samples; each push appends ``hop`` new samples and
the result for the newest frames equals the batch path applied to the buffered window.  Wraps the C++ object
behind ``b200vad_stream_*`` (device ring buffers + one CUDA graph replay per push).

With ``sincnet_packed`` the path is SincNet -> PyanNet: the hop must be a multiple of 270 samples (the SincNet frame step)
so that every push adds whole frames, and a push returns the newest ``hop // 270`` of the window's get_num_frames(window)
frames.
"""

from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib


class StreamingVad:
    def __init__(self, packed: torch.Tensor, num_layers: int = 4, num_streams: int = 256, window: int = 80000, hop: int = 160,
                 use_graph: bool = True, device: Optional[int] = None, sincnet_packed: Optional[torch.Tensor] = None):
        from .host import get_num_frames
        sinc = sincnet_packed is not None
        if sinc and (int(hop) <= 0 or int(hop) % 270):
            raise ValueError("SincNet streaming needs a hop that is a positive multiple of 270 samples (the SincNet frame step)")
        if not packed.is_cuda or (sinc and not sincnet_packed.is_cuda):
            raise _lib.B200VadError("packed weights must live on the GPU")
        self.device = packed.device.index if device is None else device
        self.packed, self.sincnet_packed = packed, sincnet_packed
        self.S, self.window, self.hop = int(num_streams), int(window), int(hop)
        self.T = get_num_frames(self.window) if sinc else (self.window + 80) // 160
        self.nf = self.hop // 270 if sinc else self.hop // 160
        h = C.c_void_p()
        if sinc:
            _lib.check(_lib.lib().b200vad_stream_create_sincnet(self.device, packed.data_ptr(), sincnet_packed.data_ptr(), num_layers,
                                                                self.S, self.window, self.hop, int(use_graph), C.byref(h)),
                       "b200vad_stream_create_sincnet")
        else:
            _lib.check(_lib.lib().b200vad_stream_create(self.device, packed.data_ptr(), num_layers, self.S, self.window, self.hop,
                                                        int(use_graph), C.byref(h)), "b200vad_stream_create")
        self._h = h
        self._prob = torch.empty((self.S, self.nf), dtype=torch.float32)
        self._dec = torch.empty((self.S, self.nf), dtype=torch.uint8)

    def push(self, chunk: torch.Tensor, thr: float = 0.5, kernel: int = 49):
        """chunk: (S, hop) float32, CPU or CUDA.  Returns (prob (S, nf), dec (S, nf), device_ms)."""
        if chunk.dtype != torch.float32 or tuple(chunk.shape) != (self.S, self.hop) or not chunk.is_contiguous():
            raise _lib.B200VadError("chunk must be a contiguous float32 tensor of shape (num_streams, hop)")
        ms = C.c_float(0)
        if chunk.is_cuda:
            torch.cuda.current_stream(chunk.device).synchronize()      # the session runs on its own stream
        _lib.check(_lib.lib().b200vad_stream_push(self._h, chunk.data_ptr(), 0 if chunk.is_cuda else 1, float(thr), int(kernel),
                                                  self._prob.data_ptr(), self._dec.data_ptr(), C.byref(ms)), "b200vad_stream_push")
        return self._prob.clone(), self._dec.clone(), ms.value

    def snapshot(self):
        """(window (S, W), prob (S, T), dec (S, T)) CPU tensors of the last push -- for parity checks."""
        w = torch.empty((self.S, self.window), dtype=torch.float32)
        p = torch.empty((self.S, self.T), dtype=torch.float32)
        d = torch.empty((self.S, self.T), dtype=torch.uint8)
        _lib.check(_lib.lib().b200vad_stream_snapshot(self._h, w.data_ptr(), p.data_ptr(), d.data_ptr()), "b200vad_stream_snapshot")
        return w, p, d

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().b200vad_stream_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
