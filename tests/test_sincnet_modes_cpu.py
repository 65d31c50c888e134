"""CPU tests of the SincNet -> PyanNet whole-path entry points: exported symbols, workspace sizing and the argument checks
that run before any CUDA call (the shared library loads without a GPU)."""
import ctypes as C

import pytest
import torch

import b200vad
from b200vad import _lib

NEW_SYMBOLS = ("b200vad_pipeline_sincnet_workspace_bytes", "b200vad_pipeline_sincnet_f32", "b200vad_pipeline_sincnet_i16",
               "b200vad_session_create_sincnet", "b200vad_stream_create_sincnet")


def test_new_symbols_exported():
    lib = _lib.lib()
    for name in NEW_SYMBOLS:
        assert hasattr(lib, name), name
        assert name in _lib.PROTOTYPES


def test_pipeline_sincnet_workspace_monotone():
    lib = _lib.lib()
    assert lib.b200vad_pipeline_sincnet_workspace_bytes(0, 128000) == 0
    assert lib.b200vad_pipeline_sincnet_workspace_bytes(4, 990) == 0          # shorter than one SincNet frame
    prev = 0
    for B in (1, 2, 37, 64, 65, 651, 652, 700, 4096):
        n = lib.b200vad_pipeline_sincnet_workspace_bytes(B, 128000)
        assert n > prev, B
        prev = n
    prev = 0
    for N in (991, 1261, 8000, 16000, 48123, 80000, 128000, 480000):
        n = lib.b200vad_pipeline_sincnet_workspace_bytes(37, N)
        assert n >= prev, N
        prev = n
    # the whole batch's layer-0 planes (B, Ts, 64) x 2 fp16 are part of it
    Ts = lib.b200vad_sincnet_num_frames(128000)
    assert lib.b200vad_pipeline_sincnet_workspace_bytes(4096, 128000) >= 4096 * Ts * 64 * 4


def test_short_waveform_refused_before_cuda():
    lib = _lib.lib()
    buf = (C.c_char * 4096)()
    p = C.addressof(buf)
    for fn in (lib.b200vad_pipeline_sincnet_f32, lib.b200vad_pipeline_sincnet_i16):
        rc = fn(p, p, 4, p, 2, 990, 990, 0.5, 49, p, p, p, p, p, 2, p, 256, None)
        assert rc == -1                                                        # B200VAD_EINVAL
        assert b"991" in lib.b200vad_last_error()
    h = C.c_void_p()
    assert lib.b200vad_session_create_sincnet(0, p, p, 4, 16, 990, C.byref(h)) == -1
    assert lib.b200vad_stream_create_sincnet(0, p, p, 4, 2, 990, 270, 0, C.byref(h)) == -1
    assert lib.b200vad_stream_create_sincnet(0, p, p, 4, 2, 16000, 160, 0, C.byref(h)) == -1   # hop not a multiple of 270
    assert lib.b200vad_stream_create_sincnet(0, p, None, 4, 2, 16000, 270, 0, C.byref(h)) == -1


def test_hop_not_multiple_of_270_refused():
    blob = torch.zeros(8, dtype=torch.uint8)
    with pytest.raises(ValueError):
        b200vad.LongFormVad(blob, 4, window=80000, hop=40000, sincnet_packed=blob)
    with pytest.raises(ValueError):
        b200vad.StreamingVad(blob, 4, num_streams=2, window=16000, hop=160, sincnet_packed=blob)
    # hop == window (reference semantics) needs no frame grid; multiples of 270 are accepted
    b200vad.LongFormVad(blob, 4, window=80000, sincnet_packed=blob)
    b200vad.LongFormVad(blob, 4, window=80000, hop=40500, sincnet_packed=blob)
    # without a SincNet blob the fbank rules stay as they were
    with pytest.raises(ValueError):
        b200vad.LongFormVad(blob, 4, window=80000, hop=40500)
