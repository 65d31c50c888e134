"""Runtime around the kernels: the host-buffer session (C++ object behind the C ABI) and the
multi-GPU plumbing (shard by utterance, gather segment lists).  One process per GPU."""

from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import torch

from . import _lib
from .host import shard_range  # noqa: F401  (re-export)


def bind_to_gpu_numa(device_index: int) -> Optional[int]:
    """Pin this process (and therefore the pinned host buffers it allocates afterwards: first touch) to the NUMA node
    the GPU hangs off.  With one process per GPU on a multi-socket host this keeps every rank's H2D copies off the
    inter-socket link.  Returns the node, or None when the topology cannot be read (then nothing is changed)."""
    import os
    try:
        props = torch.cuda.get_device_properties(device_index)
        bdf = "%04x:%02x:%02x.0" % (props.pci_domain_id, props.pci_bus_id, props.pci_device_id)
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return node
    except Exception:  # noqa: BLE001  (no sysfs / no permission: leave the affinity alone)
        return None


class _HostBlock:
    """Owner of one b200vad_host_alloc allocation (freed when the last tensor view goes away)."""

    def __init__(self, nbytes: int, write_combined: bool):
        self.ptr = _lib.lib().b200vad_host_alloc(int(nbytes), 1 if write_combined else 0)
        if not self.ptr:
            raise _lib.B200VadError("b200vad_host_alloc failed: " + (_lib.lib().b200vad_last_error() or b"").decode())
        self.buf = (C.c_char * max(int(nbytes), 1)).from_address(self.ptr)

    def __del__(self):
        try:
            if getattr(self, "ptr", None):
                _lib.lib().b200vad_host_free(self.ptr)
                self.ptr = None
        except Exception:  # noqa: BLE001  (interpreter shutdown)
            pass


def host_buffer(shape, dtype=torch.float32, write_combined: bool = False) -> torch.Tensor:
    """Page-locked host tensor from ``b200vad_host_alloc`` (optionally write-combined: write it, never read it on the CPU)."""
    n = 1
    for d in shape:
        n *= int(d)
    nbytes = n * torch.empty((), dtype=dtype).element_size()
    blk = _HostBlock(nbytes, write_combined)
    t = torch.frombuffer(blk.buf, dtype=dtype, count=n).view(*shape)
    t._b200vad_block = blk          # keeps the allocation alive as long as this tensor object
    return t


class HostSession:
    """waveforms on the HOST -> decisions / probabilities / segments on the HOST.

    Wraps ``b200vad_session_*``: the session owns device buffers for two batches in flight and
    three CUDA streams (H2D / compute / D2H).  ``run`` is the blocking form (rows are cut into
    chunks of ``chunk_rows`` and pipelined internally); ``submit`` / ``wait`` is the asynchronous
    form for a caller that streams batches.  Pass pinned tensors (``tensor.pin_memory()``).

    ``sincnet_packed`` (a ``pack_sincnet`` blob; ``packed`` then holds the D = 60 LSTM stack + head) selects the SincNet ->
    PyanNet path: ``T`` = get_num_frames(num_samples) frames per row, segments keep single-frame runs.

    ``binarize`` (a ``b200vad.Binarize``, or ``set_binarize`` later) replaces threshold / median / run-length segments by
    onset / offset hysteresis, pads and minimum durations on the mode's frame grid; ``thr`` / ``kernel`` are then ignored.
    """

    def __init__(self, packed: torch.Tensor, num_layers: int, num_samples: int, chunk_rows: int = 1024,
                 device: Optional[int] = None, sincnet_packed: Optional[torch.Tensor] = None, binarize=None):
        from .host import fbank_num_frames, get_num_frames
        from .ops import _seg_per_row
        if not packed.is_cuda or (sincnet_packed is not None and not sincnet_packed.is_cuda):
            raise _lib.B200VadError("packed weights must live on the GPU")
        self.device = packed.device.index if device is None else device
        self.packed, self.sincnet_packed = packed, sincnet_packed
        self.N = int(num_samples)
        sinc = sincnet_packed is not None
        self.T = get_num_frames(self.N) if sinc else fbank_num_frames(self.N)
        self._seg_per_row = _seg_per_row(self.T, sinc)
        self.chunk_rows = int(chunk_rows)
        h = C.c_void_p()
        if sinc:
            _lib.check(_lib.lib().b200vad_session_create_sincnet(self.device, packed.data_ptr(), sincnet_packed.data_ptr(), num_layers,
                                                                 self.chunk_rows, self.N, C.byref(h)), "b200vad_session_create_sincnet")
        else:
            _lib.check(_lib.lib().b200vad_session_create(self.device, packed.data_ptr(), num_layers, self.chunk_rows, self.N,
                                                         C.byref(h)), "b200vad_session_create")
        self._h = h
        self.binarize = None
        if binarize is not None:
            self.set_binarize(binarize)

    def set_binarize(self, binarize) -> None:
        """Post-process the following batches with ``binarize`` (a ``b200vad.Binarize``), or with threshold / median /
        run-length segments again when None.  A batch already submitted keeps its policy."""
        from .binarize import mode_step
        params = None if binarize is None else binarize.params(mode_step(self.sincnet_packed is not None)[0])
        _lib.check(_lib.lib().b200vad_session_set_binarize(self._h, params), "b200vad_session_set_binarize")
        self.binarize = binarize

    def _cap(self, B: int) -> int:
        return B * ((self.T + 1) // 2 if self.binarize is not None else self._seg_per_row)

    def run(self, wav: torch.Tensor, thr: float = 0.5, kernel: int = 49, want_dec: bool = True, want_prob: bool = False,
            out: Optional[dict] = None):
        """wav: (B, N) float32 CPU tensor.  Returns dict(dec, prob, seg) of CPU tensors."""
        if wav.is_cuda or wav.dtype != torch.float32 or wav.dim() != 2 or wav.shape[1] != self.N or not wav.is_contiguous():
            raise _lib.B200VadError("wav must be a contiguous CPU float32 tensor of shape (B, N)")
        B = wav.shape[0]
        out = out if out is not None else {}
        if want_dec and ("dec" not in out or out["dec"].shape[0] < B):
            out["dec"] = torch.empty((B, self.T), dtype=torch.uint8).pin_memory()
        if want_prob and ("prob" not in out or out["prob"].shape[0] < B):
            out["prob"] = torch.empty((B, self.T), dtype=torch.float32).pin_memory()
        cap = self._cap(B)
        if "seg_buf" not in out or out["seg_buf"].shape[0] < cap:
            out["seg_buf"] = torch.empty((max(cap, 1), 3), dtype=torch.int32).pin_memory()
        nseg = C.c_int64(0)
        _lib.check(_lib.lib().b200vad_session_run_host(
            self._h, wav.data_ptr(), B, float(thr), int(kernel),
            out["dec"].data_ptr() if want_dec else None, out["prob"].data_ptr() if want_prob else None,
            out["seg_buf"].data_ptr(), cap, C.byref(nseg)), "b200vad_session_run_host")
        out["seg"] = out["seg_buf"][: nseg.value]
        return out

    # ---- asynchronous form: two batches in flight (slot 0 / 1); PCIe copies overlap the other slot's compute
    def submit(self, slot: int, wav: torch.Tensor, thr: float = 0.5, kernel: int = 49, want_dec: bool = True,
               want_prob: bool = False, out: Optional[dict] = None) -> dict:
        """Enqueue one batch (B <= chunk_rows rows; float32 or int16 PCM samples) into ``slot`` and return at once.  ``out`` (reused across
        calls) receives pinned ``dec`` / ``prob`` buffers that are valid after ``wait(slot, out)``."""
        if wav.is_cuda or wav.dtype not in (torch.float32, torch.int16) or wav.dim() != 2 or wav.shape[1] != self.N \
                or not wav.is_contiguous():
            raise _lib.B200VadError("wav must be a contiguous CPU float32 (or int16 PCM) tensor of shape (B, N)")
        B = wav.shape[0]
        out = out if out is not None else {}
        if want_dec and ("dec" not in out or out["dec"].shape[0] != B):
            out["dec"] = torch.empty((B, self.T), dtype=torch.uint8).pin_memory()
        if want_prob and ("prob" not in out or out["prob"].shape[0] != B):
            out["prob"] = torch.empty((B, self.T), dtype=torch.float32).pin_memory()
        cap = self._cap(B)
        if "seg_buf" not in out or out["seg_buf"].shape[0] < cap:
            out["seg_buf"] = torch.empty((max(cap, 1), 3), dtype=torch.int32).pin_memory()
        out["_wav"] = wav          # keep the source alive until wait()
        fn = _lib.lib().b200vad_session_submit_host_i16 if wav.dtype == torch.int16 else _lib.lib().b200vad_session_submit_host
        _lib.check(fn(
            self._h, int(slot), wav.data_ptr(), B, float(thr), int(kernel),
            out["dec"].data_ptr() if want_dec else None, out["prob"].data_ptr() if want_prob else None),
            "b200vad_session_submit_host")
        return out

    def wait(self, slot: int, out: dict) -> dict:
        """Block until the batch submitted into ``slot`` is on the host; fills ``out['seg']``."""
        nseg = C.c_int64(0)
        buf = out["seg_buf"]
        _lib.check(_lib.lib().b200vad_session_wait(self._h, int(slot), buf.data_ptr(), buf.shape[0], C.byref(nseg)),
                   "b200vad_session_wait")
        out["seg"] = buf[: min(nseg.value, buf.shape[0])]
        out.pop("_wav", None)
        return out

    def slot_times(self, slot: int):
        """Device timeline of the slot's latest batch: ms since session creation of
        (H2D begin, H2D end, compute begin, compute end, D2H end)."""
        arr = (C.c_float * 5)()
        _lib.check(_lib.lib().b200vad_session_slot_times(self._h, int(slot), arr), "b200vad_session_slot_times")
        return list(arr)

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().b200vad_session_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def gather_segments(seg: torch.Tensor, row_base: int = 0, group=None) -> torch.Tensor:
    """All-gather per-rank segment triples (S_r, 3) int32 -> (sum S_r, 3) on every rank, rows
    re-based to global utterance ids by adding ``row_base`` to column 0.  Two collectives: one
    all_gather of the counts, one all_gather of the triples padded to max(count) (SURVEY 8e).
    Works on CUDA tensors with the NCCL backend and on CPU tensors with gloo."""
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        s = seg.clone()
        s[:, 0] += row_base
        return s
    world = dist.get_world_size(group)
    local = seg.clone()
    local[:, 0] += row_base
    n = torch.tensor([local.shape[0]], dtype=torch.int64, device=seg.device)
    counts = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(counts, n, group=group)
    counts = [int(c.item()) for c in counts]
    m = max(max(counts), 1)
    padded = torch.zeros((m, 3), dtype=torch.int32, device=seg.device)
    padded[: local.shape[0]] = local
    bufs = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(bufs, padded, group=group)
    return torch.cat([b[:c] for b, c in zip(bufs, counts)], dim=0)


class SegmentGatherer:
    """Segment-list gather that stays OFF the compute stream (SURVEY 8e: "end of corpus or every k batches, on a side stream").

    ``push(seg, seg_off, row_base)`` takes the padded output of ``torch.ops.b200vad.vad_pipeline_padded`` (nothing synchronises:
    it records an event on the current stream and returns).  The previous push is completed at that moment, while the GPU is
    already running the batch just enqueued: on a side stream the valid rows are compacted, the counts of all ranks exchanged
    with one ``all_gather_into_tensor`` and the triples with one fixed-shape ``all_gather_into_tensor`` padded to the largest
    count.  The only host reads are the 8-byte total of a batch that has already finished and the world-size counts, both on
    the side stream.  ``drain()`` completes what is pending and returns the list of gathered (S, 3) int32 tensors (global
    utterance ids in column 0), one per push, identical on every rank.  Single-process use (no process group) skips the
    collectives.  NCCL on CUDA tensors; the CPU test runs the same code over gloo with ``device="cpu"``.

    ``every=k`` batches k pushes into one exchange (SURVEY 8e's "every k batches"); ``every=0`` defers everything to
    ``drain()`` -- one exchange per corpus shard, which is what a host-driven loop wants: completing a push reads the counts
    on the host, so with one exchange per step every rank waits for the slowest rank once per step and the host cannot
    submit the next copy meanwhile (measured at 2 GPUs through the host session: 49.6 ms per step, against 39.1 ms
    without the per-step rendezvous)."""

    def __init__(self, device=None, group=None, every: int = 1):
        import torch.distributed as dist
        self.dist = dist if (dist.is_available() and dist.is_initialized()) else None
        self.group = group
        self.world = self.dist.get_world_size(group) if self.dist else 1
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.cuda = self.device.type == "cuda"
        self.side = torch.cuda.Stream(device=self.device) if self.cuda else None
        self.pending = None
        self.results = []
        self.every = int(every)
        self.batch = []

    def push(self, seg: torch.Tensor, seg_off: torch.Tensor, row_base: int = 0):
        ev = None
        if self.cuda:
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(self.device))
        if self.every != 1:
            self.batch.append((seg, seg_off, int(row_base), ev))
            if self.every > 1 and len(self.batch) >= self.every:
                self._flush_batch()
            return
        prev, self.pending = self.pending, (seg, seg_off, int(row_base), ev)
        if prev is not None:
            self._complete(prev)

    def _flush_batch(self):
        """One exchange for all batched pushes: compact each, concatenate, gather once, split back per push and rank."""
        items, self.batch = self.batch, []
        if not items:
            return
        ctx = torch.cuda.stream(self.side) if self.cuda else _NullCtx()
        with ctx:
            locs = []
            for seg, seg_off, row_base, ev in items:
                if self.cuda:
                    self.side.wait_event(ev)
                n = int(seg_off[-1].item())
                loc = seg[:n].clone()
                loc[:, 0] += row_base
                locs.append(loc)
                if self.cuda:
                    seg.record_stream(self.side)
                    seg_off.record_stream(self.side)
            if self.world == 1:
                self.results.extend(locs)
                return
            dev = items[0][0].device
            k = len(locs)
            cnt = torch.tensor([l.shape[0] for l in locs], dtype=torch.int64, device=dev)
            counts = torch.empty(self.world * k, dtype=torch.int64, device=dev)
            self.dist.all_gather_into_tensor(counts, cnt, group=self.group)
            counts = counts.reshape(self.world, k).tolist()
            m = max(max(sum(c) for c in counts), 1)
            padded = torch.zeros((m, 3), dtype=torch.int32, device=dev)
            mine = torch.cat(locs, dim=0)
            padded[: mine.shape[0]] = mine
            out = torch.empty((self.world * m, 3), dtype=torch.int32, device=dev)
            self.dist.all_gather_into_tensor(out, padded, group=self.group)
            for j in range(k):
                parts = []
                for r in range(self.world):
                    o = r * m + sum(counts[r][:j])
                    parts.append(out[o: o + counts[r][j]])
                self.results.append(torch.cat(parts, dim=0))

    def _complete(self, item):
        seg, seg_off, row_base, ev = item
        ctx = torch.cuda.stream(self.side) if self.cuda else _NullCtx()
        with ctx:
            if self.cuda:
                self.side.wait_event(ev)
            n = int(seg_off[-1].item())                       # this batch has finished; the compute stream is not touched
            local = seg[:n].clone()
            local[:, 0] += row_base
            if self.world == 1:
                self.results.append(local)
                return
            cnt = torch.tensor([n], dtype=torch.int64, device=seg.device)
            counts = torch.empty(self.world, dtype=torch.int64, device=seg.device)
            self.dist.all_gather_into_tensor(counts, cnt, group=self.group)
            counts = counts.tolist()
            m = max(max(counts), 1)
            padded = torch.zeros((m, 3), dtype=torch.int32, device=seg.device)
            padded[:n] = local
            out = torch.empty((self.world * m, 3), dtype=torch.int32, device=seg.device)
            self.dist.all_gather_into_tensor(out, padded, group=self.group)
            self.results.append(torch.cat([out[r * m: r * m + c] for r, c in enumerate(counts)], dim=0))
            if self.cuda:
                seg.record_stream(self.side)
                seg_off.record_stream(self.side)

    def drain(self):
        self._flush_batch()
        if self.pending is not None:
            prev, self.pending = self.pending, None
            self._complete(prev)
        if self.cuda:
            torch.cuda.current_stream(self.device).wait_stream(self.side)
        res, self.results = self.results, []
        return res


class _NullCtx:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False
