"""b200vad: B200-native kernels for the VAD inference hot path, behind a C ABI.

Python surface = torch.library custom ops (``torch.ops.b200vad.*``), weight packing, the
host-buffer session and the multi-GPU helpers.  The reference-shaped drop-in modules live next
to this package (``src/``, ``config/``, ``main.py``).
"""

from . import host  # noqa: F401
from ._lib import B200VadError, LIB_PATH, lib  # noqa: F401
from . import ops  # noqa: F401  (registers torch.ops.b200vad.*)
from .binarize import Binarize  # noqa: F401
from .packing import pack_model, pack_sincnet  # noqa: F401
from .runtime import HostSession, SegmentGatherer, bind_to_gpu_numa, gather_segments, host_buffer, shard_range  # noqa: F401
from . import synth  # noqa: F401
from . import score  # noqa: F401
from . import corpus  # noqa: F401
from . import manifests  # noqa: F401
from .longform import LongFormVad  # noqa: F401
from .streaming import StreamingVad  # noqa: F401

__all__ = ["ops", "host", "synth", "Binarize", "pack_model", "pack_sincnet", "HostSession", "LongFormVad", "StreamingVad", "score", "gather_segments", "SegmentGatherer", "shard_range",
           "B200VadError", "lib", "LIB_PATH"]
