"""Many recordings through LongFormVad: one list call against a loop of single-recording calls.

Workload: `--recordings` seeded synthetic recordings of uniformly 3 s .. `--max-minutes` min plus one of 1 h, made on the device
(white noise at 0.05 gated on and off at 0.05 .. 0.3 Hz, so decisions and segments are not degenerate).  Arms, for each of
{fbank -> PyanNet2, SincNet -> PyanNet} x {hop = window (reference semantics), overlapped hop} x {threshold / median, Binarize}:

  loop : [lf(w) for w in wavs]     -- one call per recording, as before the list call existed
  list : lf(wavs)                  -- one call for all of them

Both arms end in host reads of their segment triples, so a host clock around them measures finished work.  They alternate
inside every repetition (`--reps`); the report gives the median and the range.  The outputs of the two arms (prob, stream_dec,
intervals, windows of every recording) are compared for equality in the same run.  Rates are audio-hours per second of wall
time.  The card's name and power limit are read in the same run.

  python tools/longform_batch_bench.py [--recordings 500] [--max-minutes 20] [--reps 2] [--out <dir>/longform_batch.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "universal-voice-activity-detection_b200")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

import b200vad  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else q.stderr}


def recordings(n, max_minutes, dev):
    g = np.random.default_rng(2026)
    lengths = [3600 * 16000] + [int(x) for x in g.integers(3 * 16000, int(max_minutes * 60 * 16000) + 1, n)]
    gen = torch.Generator(device=dev).manual_seed(7)
    wavs = []
    for i, N in enumerate(lengths):
        t = torch.arange(N, device=dev, dtype=torch.float32) / 16000.0
        gate = (torch.sin(2 * np.pi * (0.05 + 0.25 * g.random()) * t + 6.283 * g.random()) > -0.2).float()
        wavs.append(0.05 * torch.randn(N, device=dev, generator=gen) * (0.1 + gate))
    return wavs


def models(dev):
    import oracle
    torch.manual_seed(42)
    fb = b200vad.pack_model(oracle.VadModel("PyanNet2", {"encoding_dim": 80}).eval().model.state_dict(), dev, 80, 4)
    torch.manual_seed(42)
    sd = oracle.VadModel("PyanNet", {}).eval().model.state_dict()
    sb = b200vad.pack_model({k: v for k, v in sd.items() if not k.startswith("sincnet.")}, dev, 60, 4)
    return {"fbank": (fb, None), "sincnet": (sb, b200vad.pack_sincnet(sd, dev))}


def same(a, b):
    return (a["windows"] == b["windows"] and torch.equal(a["prob"], b["prob"]) and torch.equal(a["stream_dec"], b["stream_dec"])
            and a["intervals"] == b["intervals"])


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--recordings", type=int, default=500)
    ap.add_argument("--max-minutes", type=float, default=20.0)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=None, help="write the JSON report here (outside the source tree)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("longform_batch_bench: needs a CUDA device")
    dev = torch.device("cuda:0")
    b200vad._lib.init(0)
    wavs = recordings(a.recordings, a.max_minutes, dev)
    hours = sum(w.numel() for w in wavs) / 16000 / 3600
    blobs = models(dev)
    res = {"card": card(), "recordings": len(wavs), "audio_hours": hours,
           "workload": f"1 x 1 h + {a.recordings} x U(3 s, {a.max_minutes:g} min) of gated noise, seed 2026", "arms": []}
    print(json.dumps(res["card"]), f"| {len(wavs)} recordings, {hours:.2f} h of audio", flush=True)
    pol = b200vad.Binarize(onset=0.6, offset=0.4, min_duration_on=0.2, min_duration_off=0.3, pad_onset=0.05, pad_offset=0.1)
    for front in ("fbank", "sincnet"):
        blob, sblob = blobs[front]
        for hop in (None, 270 * 120 if sblob is not None else 40000):
            for post in ("threshold_median", "binarize"):
                lf = b200vad.LongFormVad(blob, 4, hop=hop, sincnet_packed=sblob, binarize=pol if post == "binarize" else None)
                lf(wavs[1:4]); [lf(w) for w in wavs[1:4]]           # warm-up: module loads, first launches, pinned buffers
                t = {"loop": [], "list": []}
                outs = {}
                for r in range(a.reps):
                    for arm in (("loop", "list") if r % 2 == 0 else ("list", "loop")):
                        fn = (lambda: [lf(w) for w in wavs]) if arm == "loop" else (lambda: lf(wavs))
                        dt, out = wall(fn)
                        t[arm].append(dt)
                        outs.setdefault(arm, out)
                equal = all(same(x, y) for x, y in zip(outs["loop"], outs["list"]))
                row = {"front": front, "hop": hop or lf.window, "post": post, "windows": sum(o["prob"].shape[0] for o in outs["list"]),
                       "equal": equal}
                for arm in ("loop", "list"):
                    med = statistics.median(t[arm])
                    row[arm] = {"s_median": med, "s_min": min(t[arm]), "s_max": max(t[arm]), "audio_h_per_s": hours / med}
                row["speedup"] = row["loop"]["s_median"] / row["list"]["s_median"]
                res["arms"].append(row)
                print(f"{front:8s} hop {row['hop']:6d} {post:16s} {row['windows']:7d} windows | loop {row['loop']['s_median']:8.3f} s "
                      f"({row['loop']['audio_h_per_s']:7.1f} h/s) | list {row['list']['s_median']:7.3f} s "
                      f"({row['list']['audio_h_per_s']:7.1f} h/s) | x{row['speedup']:.1f} | equal {equal}", flush=True)
                del outs
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    if not all(r["equal"] for r in res["arms"]):
        sys.exit("longform_batch_bench: the list call differs from the per-recording calls")


if __name__ == "__main__":
    main()
