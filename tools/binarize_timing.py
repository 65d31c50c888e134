"""Cost of binarization (b200vad_binarize) against the default post-processing, with CUDA events.

  post-processing arms : b200vad_binarize against b200vad_threshold_median (kernel 49) + b200vad_segments (min_run 2), called
                         through the C ABI on preallocated buffers (no allocation, no host read in the timed window), at
                         4096 x 800 frames (the bench batch), 256 x 500 (the streaming shape) and one 360 000-frame stream (1 h);
  whole-path arms      : vad_pipeline_padded against vad_pipeline_binarize_padded at the bench shape (4096 x 8 s of 16 kHz noise,
                         the bench's model).

Arms alternate inside every repetition; each repetition times `--iters` back-to-back calls; the report gives the median and the
spread (min, max) over repetitions.  Probabilities of the post-processing arms are a seeded random walk over (0, 1) (runs of
speech and silence of a few frames to a few hundred); at most 13 MB, so back-to-back calls read them from L2 (both arms alike).
The card's name and power limit are read in the same run.

  python tools/binarize_timing.py [--reps 15] [--iters 20] [--out <dir>/binarize_timing.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "universal-voice-activity-detection_b200")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

import b200vad  # noqa: E402
from b200vad import _lib, synth  # noqa: E402

POLICY = dict(onset=0.6, offset=0.4, pad_onset=5, pad_offset=10, min_off=10, min_on=25)   # frames of 10 ms


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else q.stderr}


def timed(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / iters


def compare(arms, reps, iters):
    for fn in arms.values():          # warm-up: module load, first launches
        fn()
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for r in range(reps):
        order = list(arms) if r % 2 == 0 else list(arms)[::-1]
        for k in order:
            times[k].append(timed(arms[k], iters))
    return {k: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v)} for k, v in times.items()}


def postproc_arms(R, T, dev):
    L = _lib.lib()
    g = np.random.default_rng(R * 7 + T)
    steps = g.standard_normal((R, T)) * 0.15
    prob = torch.from_numpy((np.abs((np.cumsum(steps, axis=1) + 0.5) % 2.0 - 1.0)).astype(np.float32)).to(dev)
    dec = torch.empty((R, T), dtype=torch.uint8, device=dev)
    counts = torch.empty(R, dtype=torch.int32, device=dev)
    seg_off = torch.empty(R + 1, dtype=torch.int64, device=dev)
    cap = R * ((T + 1) // 2)
    seg = torch.empty((cap, 3), dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    params = _lib.BinarizeParams(**POLICY)

    def default():
        _lib.check(L.b200vad_threshold_median(prob.data_ptr(), R, T, 0.5, 49, dec.data_ptr(), 1, None, 0.0, st), "threshold_median")
        _lib.check(L.b200vad_segments(dec.data_ptr(), None, R, T, 2, counts.data_ptr(), seg_off.data_ptr(), seg.data_ptr(), cap, st),
                   "segments")

    def binarized():
        _lib.check(L.b200vad_binarize(prob.data_ptr(), None, R, T, params, dec.data_ptr(), counts.data_ptr(), seg_off.data_ptr(),
                                      seg.data_ptr(), cap, st), "binarize")

    binarized()
    torch.cuda.synchronize()
    regions = int(seg_off[R].item())
    return {"threshold_median+segments": default, "binarize": binarized}, regions


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("binarize_timing needs a CUDA device")
    dev = torch.device("cuda:0")
    _lib.init(0)
    out = {"card": card(), "policy_frames": POLICY, "reps": args.reps, "iters": args.iters, "postproc": {}}
    for R, T in ((4096, 800), (256, 500), (1, 360000)):
        arms, regions = postproc_arms(R, T, dev)
        res = compare(arms, args.reps, args.iters)
        res["regions"] = regions
        out["postproc"][f"{R}x{T}"] = res
        print(f"{R} x {T}: " + ", ".join(f"{k} {v['median_ms']:.4f} ms [{v['min_ms']:.4f}, {v['max_ms']:.4f}]"
                                          for k, v in res.items() if k != "regions") + f" ({regions} regions)", flush=True)

    from src.engines import VadModel
    torch.manual_seed(42)
    model = VadModel("PyanNet2", {"encoding_dim": 80}).eval()
    blob = b200vad.pack_model(model.model.state_dict(), dev, 80, 4)
    wav = synth.noise_batch(4096, 128000, seed=1234).to(dev)
    p = POLICY
    arms = {
        "default_step": lambda: torch.ops.b200vad.vad_pipeline_padded(wav, None, blob, 4, 0.5, 49),
        "binarized_step": lambda: torch.ops.b200vad.vad_pipeline_binarize_padded(wav, None, blob, None, 4, p["onset"], p["offset"],
                                                                                 p["pad_onset"], p["pad_offset"], p["min_off"],
                                                                                 p["min_on"]),
    }
    res = compare(arms, args.reps, 3)
    out["whole_path_4096x8s"] = res
    print("whole path 4096 x 8 s: " + ", ".join(f"{k} {v['median_ms']:.3f} ms [{v['min_ms']:.3f}, {v['max_ms']:.3f}]"
                                                 for k, v in res.items()), flush=True)
    print(json.dumps(out))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
