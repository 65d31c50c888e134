"""ctypes binding of libb200vad.so (the C ABI declared in include/b200vad.h).

The library is built in-tree by ``csrc/Makefile`` (or ``__graft_entry__.build()``) into
``b200vad/lib/libb200vad.so``.  There is no fallback: if the shared object is missing the
import of any compute entry point raises.
"""

from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# B200VAD_LIB: another build of the same library (A/B runs of compile-time kernel variants); the default is the in-tree build
LIB_PATH = os.environ.get("B200VAD_LIB") or os.path.join(_HERE, "lib", "libb200vad.so")
CSRC_DIR = os.path.normpath(os.path.join(_HERE, "..", "csrc"))

_lib = None

c_void_p, c_int, c_int64, c_size_t, c_float, c_double = C.c_void_p, C.c_int, C.c_int64, C.c_size_t, C.c_float, C.c_double

MAX_INPUT_DIM = 768     # B200VAD_MAX_INPUT_DIM: the widest LSTM input the model entry points accept



class BinarizeParams(C.Structure):
    """b200vad_binarize_params: thresholds and frame counts of the binarization (include/b200vad.h)."""
    _fields_ = [("onset", C.c_float), ("offset", C.c_float), ("pad_onset", C.c_int32), ("pad_offset", C.c_int32),
                ("min_off", C.c_int32), ("min_on", C.c_int32)]


_P_BIN = C.POINTER(BinarizeParams)

# name -> (restype, argtypes); mirrors include/b200vad.h one to one
PROTOTYPES = {
    "b200vad_abi_version": (c_int, []),
    "b200vad_last_error": (C.c_char_p, []),
    "b200vad_launch_count": (C.c_longlong, []),
    "b200vad_profile_enable": (None, [c_int]),
    "b200vad_profile_collect": (c_int, [c_int, C.POINTER(c_double), C.POINTER(c_int)]),
    "b200vad_set_impl": (c_int, [c_int]),
    "b200vad_set_lstm_tile": (c_int, [c_int]),
    "b200vad_set_lstm_fused": (c_int, [c_int]),
    "b200vad_set_lstm_pair_opt": (c_int, [c_int]),
    "b200vad_lstm_fused_clusters": (c_int, []),
    "b200vad_set_lstm_fused_debug": (c_int, [c_int, c_int]),
    "b200vad_lstm_fused_read_debug": (c_int, [c_void_p, c_int]),
    "b200vad_lstm_fused_last_timeout": (c_int, [c_void_p]),
    "b200vad_set_projection_terms": (c_int, [c_int]),
    "b200vad_set_projection_kernel": (c_int, [c_int]),
    "b200vad_set_head_fused": (c_int, [c_int]),
    "b200vad_host_alloc": (c_void_p, [c_size_t, c_int]),
    "b200vad_host_free": (None, [c_void_p]),
    "b200vad_linear_split_f32": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "b200vad_init": (c_int, [c_int]),
    "b200vad_fbank_num_frames": (c_int64, [c_int64]),
    "b200vad_fbank_f32": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p]),
    "b200vad_fbank_i16": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p]),
    "b200vad_model_packed_bytes": (c_size_t, [c_int, c_int]),
    "b200vad_model_pack_lstm": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "b200vad_model_pack_head": (c_int, [c_void_p, c_int, c_int] + [c_void_p] * 6 + [c_void_p]),
    "b200vad_model_workspace_bytes": (c_size_t, [c_int, c_int64]),
    "b200vad_model_forward_f32": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int64, c_void_p, c_void_p, c_size_t, c_void_p]),
    "b200vad_sincnet_num_frames": (c_int64, [c_int64]),
    "b200vad_sincnet_packed_bytes": (c_size_t, []),
    "b200vad_sincnet_pack": (c_int, [c_void_p] * 17 + [c_void_p]),
    "b200vad_sincnet_workspace_bytes": (c_size_t, [c_int, c_int64]),
    "b200vad_sincnet_forward_f32": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p, c_size_t, c_void_p]),
    "b200vad_median_window": (c_int, [c_double, c_double]),
    "b200vad_threshold_median": (c_int, [c_void_p, c_int, c_int64, c_float, c_int, c_void_p, c_int, c_void_p, c_float, c_void_p]),
    "b200vad_threshold_median_streams": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_float, c_int, c_void_p, c_void_p]),
    "b200vad_segments": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "b200vad_binarize": (c_int, [c_void_p, c_void_p, c_int, c_int64, _P_BIN, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "b200vad_pipeline_binarize": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int64, c_int64, _P_BIN,
                                          c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_size_t, c_void_p]),
    "b200vad_session_set_binarize": (c_int, [c_void_p, _P_BIN]),
    "b200vad_stream_set_binarize": (c_int, [c_void_p, _P_BIN]),
    "b200vad_regions_step": (c_int, [c_void_p, c_int, c_int, c_int64, _P_BIN, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "b200vad_stream_set_events": (c_int, [c_void_p, _P_BIN]),
    "b200vad_stream_end": (c_int, [c_void_p, c_void_p, c_int]),
    "b200vad_stream_events": (c_int, [c_void_p, c_void_p, c_int64, C.POINTER(c_int64)]),
    "b200vad_stat_scores": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "b200vad_score_workspace_bytes": (c_size_t, [c_int64]),
    "b200vad_score_intervals": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int64, c_int, c_void_p,
                                        c_void_p, c_void_p, c_void_p]),
    "b200vad_synth_corpus": (c_int, [c_void_p, c_int64, c_int, c_int64, C.c_uint64, c_void_p]),
    "b200vad_stitch_center": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int64, c_void_p]),
    "b200vad_stitch_center_streams": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_void_p, c_void_p]),
    "b200vad_stream_create": (c_int, [c_int, c_void_p, c_int, c_int, c_int64, c_int, c_int, C.POINTER(c_void_p)]),
    "b200vad_stream_push": (c_int, [c_void_p, c_void_p, c_int, c_float, c_int, c_void_p, c_void_p, C.POINTER(c_float)]),
    "b200vad_stream_snapshot": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "b200vad_stream_destroy": (None, [c_void_p]),
    "b200vad_pipeline_workspace_bytes": (c_size_t, [c_int, c_int64]),
    "b200vad_pipeline_fbank_f32": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int64, c_int64, c_float, c_int,
                                           c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_size_t, c_void_p]),
    "b200vad_pipeline_fbank_i16": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int64, c_int64, c_float, c_int,
                                           c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_size_t, c_void_p]),
    "b200vad_pipeline_sincnet_workspace_bytes": (c_size_t, [c_int, c_int64]),
    "b200vad_pipeline_sincnet_f32": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int64, c_int64, c_float, c_int,
                                             c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_size_t, c_void_p]),
    "b200vad_pipeline_sincnet_i16": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int64, c_int64, c_float, c_int,
                                             c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_size_t, c_void_p]),
    "b200vad_pipeline_rows": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int64, c_float, c_int, _P_BIN,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_size_t, c_void_p]),
    "b200vad_session_create_sincnet": (c_int, [c_int, c_void_p, c_void_p, c_int, c_int, c_int64, C.POINTER(c_void_p)]),
    "b200vad_stream_create_sincnet": (c_int, [c_int, c_void_p, c_void_p, c_int, c_int, c_int64, c_int, c_int, C.POINTER(c_void_p)]),
    "b200vad_session_submit_host_i16": (c_int, [c_void_p, c_int, c_void_p, c_int, c_float, c_int, c_void_p, c_void_p]),
    "b200vad_session_create": (c_int, [c_int, c_void_p, c_int, c_int, c_int64, C.POINTER(c_void_p)]),
    "b200vad_session_run_host": (c_int, [c_void_p, c_void_p, c_int, c_float, c_int, c_void_p, c_void_p, c_void_p, c_int64,
                                         C.POINTER(c_int64)]),
    "b200vad_session_submit_host": (c_int, [c_void_p, c_int, c_void_p, c_int, c_float, c_int, c_void_p, c_void_p]),
    "b200vad_session_wait": (c_int, [c_void_p, c_int, c_void_p, c_int64, C.POINTER(c_int64)]),
    "b200vad_session_slot_times": (c_int, [c_void_p, c_int, C.POINTER(c_float)]),
    "b200vad_session_destroy": (None, [c_void_p]),
}


class B200VadError(RuntimeError):
    pass


def lib() -> C.CDLL:
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B200VadError(
                f"{LIB_PATH} is missing: build it with `make -C {CSRC_DIR}` (or __graft_entry__.build()). "
                "There is no CPU / PyTorch fallback for this path."
            )
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(handle, name)          # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().b200vad_last_error()
        extra = ""
        try:   # a bounded wait of the fused LSTM kernel that timed out leaves its last words in page-locked host memory
            rec = (C.c_int * 7)()
            lib().b200vad_lstm_fused_last_timeout(rec)
            if rec[0]:
                extra = (f" [lstm_fused wait timed out: block {rec[1]} thread {rec[2]} (warp {rec[2] // 32}) site {rec[3]} "
                         f"barrier 0x{rec[4] & 0xffffffff:x} parity {rec[5]} grid {rec[6]}]")
        except Exception:  # noqa: BLE001
            pass
        raise B200VadError(f"{what} failed (code {rc}): {msg.decode() if msg else '?'}{extra}")


_inited = set()


def init(device_index: int) -> None:
    if device_index not in _inited:
        check(lib().b200vad_init(device_index), "b200vad_init")
        _inited.add(device_index)
