#!/usr/bin/env python
"""bench.py -- audio-hours/sec of the VAD inference hot path (fbank + PyanNet2 forward +
threshold/median + segments) on N B200s of one node.

Workload (BASELINE.json configs[1]): a batch of 4096 x 8 s synthetic 16 kHz utterances per GPU
(random-init PyanNet2, seed 42).  One "step" = one pass of the whole path over that batch.
  value : whole-job audio-hours/sec with the waveforms already resident in HBM
          (torch.ops.b200vad.vad_pipeline on device buffers), CUDA events, max over ranks.
  e2e   : the same metric through the host-facing C ABI (b200vad_session_submit_host / _wait):
          waveforms in PINNED HOST memory, H2D copy of every step's input and D2H of its results
          inside the timed region; a step's batch is submitted as two sub-batches of 2048 rows (B200VAD_BENCH_SUB) and two
          submissions are in flight, so every copy overlaps the compute of the previous sub-batch and only the last
          sub-batch's compute (13 ms, not 29) is exposed.
  roofline : the dominant kernel (the fused LSTM layer kernel: input projection + recurrence), timed live with
          CUDA events on its own stream inside the timed region (b200vad_profile_*).  SURVEY 8(d) bounds the
          LSTM by the TENSOR pipe: frac = algorithmic FLOPs per launch / measured duration / sustained bf16 peak;
          path_frac = the same for the whole model over the whole step; traffic from the committed ncu capture.
  pyannet  : the SincNet path (PyanNet through the drop-in VadModel) on the same 4096 x 8 s batch.
  modes    : BASELINE configs 1 / 3 / 5 and a sharded corpus run (config 4) at this build (N = 1 only).
  cpu_baseline : the oracle (CPU restatement of the reference path) on a bounded sample, rank 0, N=1.
`--impl reference` times the reference's CPU implementation of the path (the oracle port) instead, on the same
`config.workload` (a bounded sample of its rows per step).
`--dump-outputs DIR` writes what the last timed step of the device-resident arm returned (rank 0's probabilities, decisions and
per-row segment counts, and the gathered segment list) as DIR/<name>.npy, so that two builds can be compared output for output:
the inputs and weights are seeded, identical from run to run.
Multi-GPU: `torchrun --nproc-per-node N bench.py --gpus N ...`; utterances are sharded across ranks (no data-path
collective); segment lists are gathered with NCCL on a side stream, one step behind the compute (b200vad.SegmentGatherer),
and drained inside the timed region; scaling = weak.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "universal-voice-activity-detection_b200"))
sys.path.insert(0, ROOT)

METRIC = "audio-hours/sec (fbank+VAD fwd)"
UNIT = "audio-hours/s"
ROWS, SECONDS = 4096, 8.0
N_SAMPLES = int(SECONDS * 16000)
T_FRAMES = (N_SAMPLES + 80) // 160
# Per-kernel algorithmic work per FRAME (10 ms of one utterance; 3 276 800 frames per launch at 4096 x 8 s), DESIGN.md
# section 4.  `traffic` = dram__bytes_read.sum + dram__bytes_write.sum per launch of an `ncu --set full` capture at the named
# workload (profiles/r02_ncu_full_summary.md; average over the launches of a kind).  `executed_over_algorithmic`: the
# split-precision products execute 3 (layer-0 input product, head) / 2 (everything else) fp16 MMAs per algorithmic one.
LSTM_FLOP = [2 * 2 * 512 * (80 + 128)] + [2 * 2 * 512 * (256 + 128)] * 3          # per frame and layer, both directions
LSTM_EXEC = [2 * 2 * 512 * (3 * 80 + 2 * 128)] + [2 * 2 * 512 * 2 * (256 + 128)] * 3
KERNELS = {
    0: {"name": "lstm_fused_kernel (input projection + recurrence per layer, 4 launches/step)", "bound": "tensor", "tensor": True,
        # per layer: x planes read 2 x 2 B x D (320 B layer 0, 1024 B layers 1-3) + y planes written 1024 B; no xg tensor.
        # Measured traffic is 1.45x that: the forward and the backward sweep of a layer each read x (they meet only at T/2, and
        # 3.3 GB of x per layer does not stay in the 126 MB L2); the y planes are written exactly once (3.33 GB per launch).
        "bytes_per_frame": ((320 + 1024) + 3 * (1024 + 1024)) / 4.0, "flop_per_frame": sum(LSTM_FLOP) / 4.0,
        "executed_over_algorithmic": sum(LSTM_EXEC) / float(sum(LSTM_FLOP)),
        "traffic": (5.384654e9 + 10.010359e9 + 10.006204e9 + 10.014153e9) / 4},
    1: {"name": "gemm_xg_pair_kernel (legacy input projections, b200vad_set_lstm_fused(0) only)", "bound": "hbm", "tensor": True,
        "bytes_per_frame": (3 * (1024 + 4096) + (320 + 4096)) / 4.0, "flop_per_frame": 2 * 1024 * (3 * 256 + 80) / 4.0,
        "executed_over_algorithmic": (3 * 80 + 2 * 3 * 256) / (80 + 3 * 256.0), "traffic": (14.76e9 + 3 * 16.76e9) / 4},
    2: {"name": "head_fused_kernel (head linears + classifier + sigmoid, 1 launch/step)", "bound": "hbm", "tensor": True,
        # y planes 1024 B read -> 4 B probability (the hidden activations stay in shared memory)
        "bytes_per_frame": 1024 + 4, "flop_per_frame": 2 * (256 * 128 + 128 * 128),
        "executed_over_algorithmic": 3.0, "traffic": 3.372568e9},
    3: {"name": "fbank_kernel (frame/window/FFT/mel/log, 1 launch/step)", "bound": "hbm", "tensor": False,
        "bytes_per_frame": 640 + 320, "flop_per_frame": 55000, "executed_over_algorithmic": 1.0, "traffic": 3.122489e9},
}
MODEL_FLOP_PER_FRAME = 2.884e6
ALGORITHMIC_BYTES_PER_AUDIO_S = 64.4e3      # SURVEY 8(d): 64 000 (waveform f32) + 400 (probabilities)
# DRAM traffic of one step at the named workload, summed over all 10 launches of the ncu --set full capture
# (profiles/r02_ncu_full_summary.md): row_sum 2.10 + fbank 3.12 + 4 x lstm_fused 35.42 + head 3.37 + post 0.02 GB.  The 20.9x over
# the algorithmic bytes is the five inter-kernel tensors (fbank features, four layers' y planes as two fp16 planes each) that
# leave the chip once and come back 1-2 times; see DESIGN.md section 4 for why they cannot stay in the 126 MB L2.
STEP_TRAFFIC_BYTES = 44.029487e9
WORKLOAD = (f"{ROWS} x {SECONDS:.0f} s synthetic 16 kHz utterances per GPU: fbank + PyanNet2 (4xBiLSTM128, random-init seed 42) "
            "forward + threshold/median(49) + segments")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d["bf16_tflops_sustained"], "src": "measured"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "src": "fallback"}


DUMP_BYTES = 64 << 20


def dump_outputs(dirname, arrays):
    """Writes each array as DIR/<name>.npy: integers wider than 16 bits as float64, everything else as float32 (both exact
    for the outputs of the path).  Each array gets an equal share of DUMP_BYTES; one larger than that is replaced by a fixed,
    seeded sample of its rows, sorted, whose row indices are written as DIR/<name>_rows.npy."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    share = DUMP_BYTES // len(arrays) - 1024          # room for the .npy headers
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        a = a.astype(np.float64 if a.dtype.kind in "iu" and a.dtype.itemsize > 2 else np.float32)
        rows_path = os.path.join(dirname, f"{name}_rows.npy")
        if a.nbytes > share:
            per_row = a.nbytes // a.shape[0] + 8
            idx = np.sort(np.random.default_rng(0).choice(a.shape[0], share // per_row, replace=False))
            a = a[idx]
            np.save(rows_path, idx.astype(np.float64))
        elif os.path.exists(rows_path):
            os.remove(rows_path)
        np.save(os.path.join(dirname, f"{name}.npy"), a)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 50 ms while the timed regions (device arm and e2e arm) run."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:  # noqa: BLE001
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference(sample_rows, steps, warmup, threads):
    """The reference path on the host cores (oracle port): fbank -> PyanNet2 -> where/medfilt -> Python RLE."""
    import torch
    import oracle
    from b200vad import synth
    torch.set_num_threads(threads)
    torch.manual_seed(42)
    model = oracle.VadModel("PyanNet2", {"encoding_dim": 80}).eval()
    wav = synth.noise_batch(sample_rows, N_SAMPLES, seed=1234)

    def step():
        with torch.no_grad():
            feats = oracle.lhotse_fbank(wav)
            dec = model.predict_step({"inputs": feats}).squeeze(-1)
        segs = [oracle.rle_segments(dec[i].tolist(), 0.01) for i in range(dec.shape[0])]
        return segs

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return (sample_rows * SECONDS / 3600.0) / dt, dt


def run_reference(args, out):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    sample_rows = 128
    steps, warmup = max(1, args.steps), max(1, args.warmup)
    value, dt = cpu_reference(sample_rows, steps, warmup, threads)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "rows_per_gpu": ROWS, "samples_per_row": N_SAMPLES, "frames_per_row": T_FRAMES,
                       "sample": f"{sample_rows} of the {ROWS} rows per step (CPU arm: bounded sample of the same workload)"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": f"{sample_rows} x {SECONDS:.0f} s utterances per step, torch CPU threads={threads}"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    out.emit(json.dumps(line))
    return 0


def other_paths(torch, b200vad, VadModel, dev, blob, wav_dev, rows):
    """The other named paths at this build, on the GPU the bench line ran on (CUDA events; parity for each lives in tests/):
    `pyannet`: the SincNet front-end + LSTM head (PyanNet through the drop-in VadModel) on the bench batch;
    `modes`: BASELINE configs 1 (60 s clip as 12 reference windows through the drop-in modules), 3 (1 h long-form, reference
    window semantics), 5 (256 streams x 5 s ring x 10 ms hop, per-push latency) and 4 (sharded corpus: here 50 h on this GPU)."""
    from b200vad import corpus
    from src.features import Fbank, FbankConfig
    from src.scripts.predict import get_segments

    def timed(fn, iters, warm):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    out = {}
    # ---- PyanNet (north_star's SincNet front-end) on the same batch
    torch.manual_seed(42)
    pm = VadModel("PyanNet", {}).eval().to(dev)
    with torch.no_grad():
        ms_all = timed(lambda: pm.predict_step({"inputs": wav_dev}, 0), 5, 3)
        ms_front = timed(lambda: pm.model.sincnet.frames_time_major(wav_dev.unsqueeze(1)), 5, 2)
    hours = rows * SECONDS / 3600.0
    ts = int(b200vad.lib().b200vad_sincnet_num_frames(N_SAMPLES))
    out["pyannet"] = {"value": hours / (ms_all / 1e3), "unit": UNIT, "ms_per_step": ms_all, "frontend_ms": ms_front,
                      "workload": f"{rows} x {SECONDS:.0f} s through VadModel('PyanNet').predict_step: SincNet (sinc conv 251/10 + 2 x conv5, "
                                  f"MaxPool3 + InstanceNorm + LeakyReLU) -> 4 x BiLSTM(128) -> head -> median(49); {ts} frames per row",
                      "roofline": {"bound": "tensor", "frontend_flop_per_audio_s": 96.3e6, "head_flop_per_audio_s": 168.5e6,
                                   "achieved_tflops": (96.3e6 + 168.5e6) * rows * SECONDS / (ms_all / 1e3) / 1e12,
                                   "note": "algorithmic FLOPs (SURVEY 8d) over the whole PyanNet step"}}
    del pm
    modes = {}
    # ---- config 1
    torch.manual_seed(42)
    model = VadModel("PyanNet2", {"encoding_dim": 80}).eval().to(dev)
    clip = b200vad.synth.meeting_batch(1, 960000, seed=42)[0].to(dev)
    fb = Fbank(FbankConfig(device="cuda"))

    def config1():
        with torch.no_grad():
            dec = model.predict_step({"inputs": fb.extract_batch(clip.view(12, 80000), 16000)}, 0)
        return get_segments(dec, [60.0], 0.01)
    modes["config1_60s_clip_ms"] = timed(config1, 10, 2)
    # ---- config 3
    g = torch.Generator(device=dev).manual_seed(1)
    wav = 0.05 * torch.randn(3600 * 16000, device=dev, generator=g)
    lf = b200vad.LongFormVad(blob, 4, hop=None)
    modes["config3_one_hour_720_windows_ms"] = timed(lambda: lf(wav), 3, 1)
    lf2 = b200vad.LongFormVad(blob, 4, hop=40000)
    modes["config3_one_hour_overlap_1439_windows_ms"] = timed(lambda: lf2(wav), 3, 1)
    del wav, lf, lf2
    # ---- config 5
    sv = b200vad.StreamingVad(blob, 4, num_streams=256, window=80000, hop=160)
    gen = torch.Generator().manual_seed(0)
    chunks = [(0.1 * torch.randn(256, 160, generator=gen)).pin_memory() for _ in range(16)]
    dms = []
    for i in range(330):
        _, _, ms = sv.push(chunks[i % 16])
        if i >= 30:
            dms.append(ms)
    sv.close()
    dms.sort()
    modes["config5_streaming_256x5s_push_ms_p50"] = dms[len(dms) // 2]
    modes["config5_streaming_256x5s_push_ms_p99"] = dms[min(len(dms) - 1, int(0.99 * len(dms)))]
    # ---- config 4 (one rank's share of a sharded corpus: waveforms synthesised on the device per batch, segment gather at the end)
    corpus_hours = 50.0
    U = int(round(corpus_hours * 3600 / SECONDS))
    corpus.run_corpus(blob, 4096, N_SAMPLES, 0, 1, 4096)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    seg, _ = corpus.run_corpus(blob, U, N_SAMPLES, 0, 1, 4096)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    modes["corpus_audio_h_s"] = corpus_hours / dt
    modes["corpus_note"] = f"{corpus_hours:g} h = {U} x 8 s utterances on this GPU incl. on-device synthesis and the final segment gather ({int(seg.shape[0])} segments)"
    out["modes"] = modes
    return out


class _OnlyJsonOnStdout:
    """Libraries (NCCL's version banner, warnings) may write to fd 1; the contract is ONE JSON line on stdout.
    Everything else is diverted to stderr until `emit` writes the line to the real stdout."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, line: str):
        sys.stdout.flush()
        os.write(self.real, (line + "\n").encode())


def main():
    jout = _OnlyJsonOnStdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=ROWS, help="utterances per GPU per step (default = the named workload)")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-modes", action="store_true", help="skip the PyanNet arm and the configs 1 / 3 / 4 / 5 timings")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (at most 64 MB; b200 path only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    if args.impl == "reference":
        return run_reference(args, jout)

    import torch
    import torch.distributed as dist
    import b200vad
    from b200vad import _lib, synth
    from src.engines import VadModel
    import ctypes as C

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the b200 path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = b200vad.bind_to_gpu_numa(local)      # pinned host buffers land on the GPU's own NUMA node
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    warmup = max(args.warmup, 3)
    steps = args.steps
    rows = args.rows
    L = _lib.lib()

    torch.manual_seed(42)
    model = VadModel("PyanNet2", {"encoding_dim": 80}).eval()
    blob = b200vad.pack_model(model.model.state_dict(), dev, 80, 4)
    # this rank's shard of the global utterance list (weak scaling: `rows` per GPU)
    lo, hi = b200vad.shard_range(rows * world, rank, world)
    wav_host = synth.noise_batch(hi - lo, N_SAMPLES, seed=1234 + rank, pin=True)
    wav_dev = wav_host.to(dev)
    host_mem = "pinned (cudaHostAlloc via torch)"
    if os.environ.get("B200VAD_BENCH_WC", "0") == "1":
        # write-combined pinned staging buffer (b200vad_host_alloc): written once by the producer, read only by the GPU's DMA
        wc = b200vad.host_buffer(tuple(wav_host.shape), torch.float32, write_combined=True)
        wc.copy_(wav_host)
        wav_host = wc
        host_mem = "pinned write-combined (b200vad_host_alloc)"
    hours_step_global = rows * world * SECONDS / 3600.0

    # segment lists: fixed-capacity device output (no host sync in the step), gathered across ranks one step behind the
    # compute on a side stream and drained inside the timed region (SURVEY 8e)
    gatherer = b200vad.SegmentGatherer(device=dev)

    def device_step():
        prob, dec, seg, counts, seg_off = torch.ops.b200vad.vad_pipeline_padded(wav_dev, None, blob, 4, 0.5, 49)
        gatherer.push(seg, seg_off, row_base=lo)
        return prob, dec, counts

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident arm
    for _ in range(warmup):
        device_step()
    gatherer.drain()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = L.b200vad_launch_count()
    L.b200vad_profile_enable(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    # only the last step's outputs are kept: each earlier step's are released at once, so every step reuses the same buffers
    for _ in range(steps - 1):
        device_step()
    last = device_step()
    gathered = gatherer.drain()                 # completes the pending gathers; the compute stream waits for the side stream
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    nseg_gathered = int(gathered[-1].shape[0]) if gathered else 0
    launches = L.b200vad_launch_count() - launches0
    prof = {}
    for kind in KERNELS:
        tot_ms, nl = C.c_double(0), C.c_int(0)
        _lib.check(L.b200vad_profile_collect(kind, C.byref(tot_ms), C.byref(nl)), "profile_collect")
        prof[kind] = (tot_ms.value, nl.value)
    L.b200vad_profile_enable(0)
    if args.dump_outputs and rank == 0:
        prob, dec, counts = last
        dump_outputs(args.dump_outputs, {"prob": prob, "dec": dec, "counts": counts, "segments": gathered[-1]})
    del last
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = t.item() / steps
    value = hours_step_global / (ms_per_step / 1e3)

    # ---------------- end-to-end arm (host buffers through the C ABI session)
    # streaming form of the host API: submit(slot) enqueues H2D + path + D2H of one step's batch, wait(slot)
    # returns its host results.  Two steps are in flight, so step i+1's H2D overlaps step i's compute; every
    # step's copies are inside the timed region (pipeline fill and drain included).
    # A step's batch goes through the session as `sub` equal sub-batches (two in flight): the H2D copy of a sub-batch overlaps the
    # compute of the previous one INSIDE the step as well, so the part of the pipeline that cannot overlap (the last compute) is a
    # sub-batch, not a batch.  Every byte of every step is still copied inside the timed region.
    sub = max(1, int(os.environ.get("B200VAD_BENCH_SUB", "2")))
    while (hi - lo) % sub:
        sub -= 1
    sub_rows = (hi - lo) // sub
    sess = b200vad.HostSession(blob, 4, N_SAMPLES, chunk_rows=sub_rows, device=local)
    outs = [{}, {}]
    # host-driven loop: the segment lists of all steps are exchanged ONCE, at the drain inside the timed region (a per-step
    # exchange makes the host wait for the slowest rank every step, and the next H2D cannot be submitted meanwhile)
    e2e_gatherer = b200vad.SegmentGatherer(device=dev, every=0)

    def e2e_finish(slot, j):
        res = sess.wait(slot, outs[slot])
        seg = res["seg"]
        if world > 1:
            # host segment list of this sub-batch -> device -> side-stream gather (completed at the drain)
            sd = seg.to(dev, non_blocking=True)
            off = torch.tensor([0, sd.shape[0]], dtype=torch.int64, device=dev)
            e2e_gatherer.push(sd, off, row_base=lo + j * sub_rows)
        return seg

    def e2e_run(k):
        """k steps = k * sub submissions; returns the segments of the LAST step (all its sub-batches)"""
        counts = []
        n = k * sub
        for i in range(n):
            j = i % sub
            outs[i & 1] = sess.submit(i & 1, wav_host[j * sub_rows:(j + 1) * sub_rows], 0.5, 49, want_dec=True, want_prob=False,
                                      out=outs[i & 1])
            if i >= 1:
                counts.append(e2e_finish((i - 1) & 1, (i - 1) % sub).shape[0])
        counts.append(e2e_finish((n - 1) & 1, (n - 1) % sub).shape[0])
        e2e_gatherer.drain()
        return sum(counts[-sub:])

    e2e_run(2)
    barrier()
    t0 = time.perf_counter()
    e0.record()
    nseg = e2e_run(steps)
    e1.record()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    # wait() blocks on the last D2H, so host wall time and device events bracket the same region
    t = torch.tensor([max(e0.elapsed_time(e1), wall_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = t.item() / steps
    e2e_value = hours_step_global / (e2e_ms / 1e3)
    # device timeline of the last two batches of this rank (CUDA events inside the session): where an e2e step goes
    st = [sess.slot_times(sl) for sl in (0, 1)]
    slot_ms = {"h2d": round(sum(x[1] - x[0] for x in st) / 2, 3), "h2d_to_compute_gap": round(sum(x[2] - x[1] for x in st) / 2, 3),
               "compute": round(sum(x[3] - x[2] for x in st) / 2, 3), "d2h": round(sum(x[4] - x[3] for x in st) / 2, 3),
               "note": "rank 0, mean of the last two submissions (sub-batches): H2D copy, wait for the compute stream, device path, D2H of the results"}
    clocks = sampler.stop() if rank == 0 else None
    # informational: the same loop fed 16-bit PCM (half the PCIe bytes, identical results -- tests/test_gpu_edges.py); the
    # headline e2e above keeps the reference's float32 waveforms
    pcm_host = (wav_host * 32768.0).clamp_(-32768, 32767).to(torch.int16).pin_memory()
    wav_keep, wav_host = wav_host, pcm_host
    e2e_run(2)
    barrier()
    t0 = time.perf_counter()
    e2e_run(steps)
    barrier()
    t = torch.tensor([(time.perf_counter() - t0) * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    pcm_ms = t.item() / steps
    wav_host = wav_keep
    h2d = wav_host.numel() * 4
    d2h = (hi - lo) * T_FRAMES + nseg * 12 + 8
    sess.close()

    # ---------------- copy-only H2D probe (what bounds e2e with float32 host waveforms): all ranks copy at the same time
    probe_dst = torch.empty_like(wav_dev)
    for _ in range(2):
        probe_dst.copy_(wav_host, non_blocking=True)
    barrier()
    e0.record()
    for _ in range(5):
        probe_dst.copy_(wav_host, non_blocking=True)
    e1.record()
    barrier()
    h2d_gbs = 5 * h2d / (e0.elapsed_time(e1) / 1e3) / 1e9
    t = torch.tensor([h2d_gbs, h2d_gbs], dtype=torch.float64, device=dev)
    if world > 1:
        tmin = t.clone()
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        h2d_min, h2d_sum = tmin[0].item(), t[1].item()
    else:
        h2d_min = h2d_sum = h2d_gbs
    del probe_dst
    h2d_floor_ms = h2d / (h2d_min * 1e9) * 1e3            # the slowest rank's copy time of one step's input

    # ---------------- informational: the device-resident step with two batches in flight on two compute streams (the next batch's
    # fbank / head run on the 16 SMs the 33 LSTM clusters leave idle and in the wave tails).  The headline `value` keeps one stream:
    # its per-kernel CUDA-event timings (roofline) need kernels that do not wait for another stream's work.
    two_streams = None
    if world == 1 and not args.skip_modes:
      try:
        ss = [torch.cuda.Stream(device=dev) for _ in range(2)]
        keep = [None, None]

        def ts_step(i):
            with torch.cuda.stream(ss[i & 1]):
                keep[i & 1] = torch.ops.b200vad.vad_pipeline_padded(wav_dev, None, blob, 4, 0.5, 49)

        for i in range(4):
            ts_step(i)
        torch.cuda.synchronize()
        e0.record()
        for st_ in ss:
            st_.wait_event(e0)
        for i in range(steps):
            ts_step(i)
        for st_ in ss:
            torch.cuda.current_stream().wait_stream(st_)
        e1.record()
        torch.cuda.synchronize()
        ts_ms = e0.elapsed_time(e1) / steps
        two_streams = {"value": hours_step_global / (ts_ms / 1e3), "unit": UNIT, "ms_per_step": ts_ms,
                       "note": "same device-resident step, batches alternating over two CUDA streams (informational)"}
        del keep, ss
        torch.cuda.empty_cache()          # two more 21 GB workspaces sit in the allocator's per-stream pools; the C-side sessions below use cudaMalloc
      except Exception as exc:  # noqa: BLE001 -- informational
        two_streams = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        print(f"bench.py: the two-stream arm failed: {exc}", file=sys.stderr)

    # ---------------- the SincNet path (PyanNet) and the other BASELINE configs at this build (single GPU only)
    extra = {}
    if world == 1 and not args.skip_modes:
        try:
            extra = other_paths(torch, b200vad, VadModel, dev, blob, wav_dev, rows)
        except Exception as exc:  # noqa: BLE001 -- informational arms must not cost the headline line
            extra = {"modes_error": f"{type(exc).__name__}: {exc}"[:300]}
            print(f"bench.py: the informational arms failed: {exc}", file=sys.stderr)

    if rank == 0:
        peaks = load_peaks()
        frames_per_launch = T_FRAMES * (hi - lo)
        kernels = {}
        for k, (tms, n) in prof.items():
            spec = KERNELS[k]
            if tms <= 0 or n == 0:
                continue
            ent = {"launches": n, "avg_launch_ms": tms / n, "share_of_step": tms / (ms_per_step * steps)}
            gbs = spec["bytes_per_frame"] * frames_per_launch * n / (tms / 1e3) / 1e9
            tfs = spec["flop_per_frame"] * frames_per_launch * n / (tms / 1e3) / 1e12
            ent["algorithmic_bytes_per_frame"] = spec["bytes_per_frame"]
            ent["algorithmic_flop_per_frame"] = spec["flop_per_frame"]
            ent["hbm_gbs"] = gbs
            ent["hbm_frac"] = gbs / peaks["hbm_gbs"]
            ent["tflops"] = tfs
            ent["tensor_frac"] = tfs * spec["executed_over_algorithmic"] / peaks["tf_sustained"] if spec["tensor"] else None
            ent["bound"] = spec["bound"]
            ent["traffic"] = spec["traffic"] if rows == ROWS else None      # captured at the named workload only
            kernels[spec["name"]] = ent
        dom = max(prof, key=lambda k: prof[k][0])
        dspec, (tms, n) = KERNELS[dom], prof[dom]
        dent = kernels[dspec["name"]]
        whole_tf = MODEL_FLOP_PER_FRAME * frames_per_launch / (ms_per_step / 1e3) / 1e12
        alg_bytes_step = ALGORITHMIC_BYTES_PER_AUDIO_S * (hi - lo) * SECONDS
        if dspec["bound"] == "hbm":
            roof = {"kernel": dspec["name"], "bound": "hbm", "achieved": dent["hbm_gbs"], "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": dent["hbm_frac"], "traffic": dent["traffic"],
                    "peak_source": f"{peaks['src']} copy bandwidth (MEASURED_PEAKS.json hbm_gbs)"}
        else:
            # SURVEY 8(d): the LSTM is bounded by the tensor pipe; achieved counts ALGORITHMIC FLOPs (2 * 512 * (D + 128) per
            # frame, layer and direction), the split-precision products execute 2-3 fp16 MMAs per algorithmic one (executed_frac)
            roof = {"kernel": dspec["name"], "bound": "tensor", "achieved": dent["tflops"], "peak": peaks["tf_sustained"],
                    "unit": "TFLOP/s", "frac": dent["tflops"] / peaks["tf_sustained"], "traffic": dent["traffic"],
                    "executed_frac": dent["tensor_frac"],
                    "peak_source": f"{peaks['src']} bf16 dense sustained (MEASURED_PEAKS.json bf16_tflops_sustained)"}
        roof.update({"launches": int(n), "avg_launch_ms": tms / max(n, 1), "share_of_step": dent["share_of_step"],
                     "algorithmic_per_launch": "FLOPs (bytes) per frame below x 3 276 800 frames per launch (DESIGN.md section 4)",
                     "path_frac": whole_tf / peaks["tf_sustained"], "path_tflops": whole_tf,
                     "path_note": "whole model (2.884 MFLOP per frame, SURVEY 8d) over the whole step vs the sustained tensor peak",
                     "step_traffic_bytes": STEP_TRAFFIC_BYTES if rows == ROWS else None,
                     "algorithmic_bytes_per_step": alg_bytes_step,
                     "traffic_over_algorithmic": (STEP_TRAFFIC_BYTES / alg_bytes_step) if (STEP_TRAFFIC_BYTES and rows == ROWS) else None,
                     "kernels": kernels})
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 operands / f32 accumulate (fbank, activations, cell state in f32)", "data": "synthetic",
            "config": {"workload": WORKLOAD if rows == ROWS else WORKLOAD.replace(str(ROWS), str(rows), 1), "rows_per_gpu": rows, "samples_per_row": N_SAMPLES,
                       "frames_per_row": T_FRAMES, "parallelism": f"utterance-sharded x{world}",
                       "l2": f"inputs ({rows * N_SAMPLES * 4 / 1e9:.2f} GB waveforms + GBs of intermediates per step) exceed the 126 MB L2; no explicit flush"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms, "host_numa_node": numa, "host_memory": host_mem,
                    "h2d_ceiling_gbs": {"per_gpu_min": h2d_min, "aggregate": h2d_sum,
                                        "note": "copy-only H2D of the same pinned batch, all ranks at once, CUDA events"},
                    "h2d_floor_ms_per_step": h2d_floor_ms, "e2e_over_h2d_floor": h2d_floor_ms / e2e_ms,
                    "slot_ms": slot_ms,
                    "pcm16_input": {"value": hours_step_global / (pcm_ms / 1e3), "ms_per_step": pcm_ms, "h2d_bytes_per_step": h2d // 2,
                                    "note": "same API fed int16 PCM host waveforms (b200vad_session_submit_host_i16); informational"},
                    "sub_batches_per_step": sub,
                    "api": f"b200vad_session_submit_host / b200vad_session_wait: each step's {hi - lo} rows as {sub} sub-batch(es) of {sub_rows}, "
                           "two submissions in flight (pinned host waveforms -> host decisions + segments)"},
            "gpu_launches": int(launches),
            "roofline": roof,
            "whole_model_tflops": whole_tf,
            "segments_gathered_per_step": nseg_gathered,
            "clocks": clocks,
        }
        line.update(extra)
        if two_streams:
            line["two_streams"] = two_streams
        if world == 1 and not args.skip_cpu_baseline:
            threads = os.cpu_count() or 1
            try:
                v, dt = cpu_reference(512, 1, 1, threads)
                line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                                        "sample": f"512 x {SECONDS:.0f} s utterances (oracle: torch CPU fbank + nn.LSTM + scipy medfilt + Python RLE), {dt:.1f} s/step"}
            except Exception as exc:  # noqa: BLE001 -- the GPU line is still worth printing
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": threads, "kind": "port", "sample": f"failed: {type(exc).__name__}: {exc}"[:300]}
        jout.emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
