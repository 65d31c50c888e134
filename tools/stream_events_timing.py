"""Cost of streaming speech events (b200vad_stream_set_events / b200vad_regions_step), with CUDA events.

  push arms   : the config-5 streaming session (256 streams, 5 s windows, 160-sample hop, CUDA graph) with events off and on,
                the bench's model and chunks; the arms alternate three times in one process, each timing `--pushes` pushes
                after 30 warm-up pushes (device ms per push as StreamingVad.push reports it: H2D copy, graph, D2H copies);
  kernel arms : b200vad_regions_step alone on preallocated buffers at 256 x 1 frames (one 10 ms hop) and 256 x 500 (a hop
                as long as the window), `--iters` back-to-back launches between two CUDA events, repeated `--reps` times.

The card's name and power limit are read in the same run.

  python tools/stream_events_timing.py [--pushes 300] [--iters 1000] [--reps 5] [--out <dir>/stream_events_timing.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "universal-voice-activity-detection_b200")]

import torch  # noqa: E402

import b200vad  # noqa: E402
from b200vad import _lib  # noqa: E402

POLICY = dict(onset=0.6, offset=0.4, min_duration_on=0.25, min_duration_off=0.1, pad_onset=0.05, pad_offset=0.1)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else q.stderr}


def pct(v, q):
    v = sorted(v)
    return v[min(len(v) - 1, int(q * len(v)))]


def push_arm(blob, events, chunks, pushes):
    sv = b200vad.StreamingVad(blob, 4, num_streams=256, window=80000, hop=160,
                              events=b200vad.Binarize(**POLICY) if events else None)
    ms, n_ev = [], 0
    for i in range(30 + pushes):
        _, _, t = sv.push(chunks[i % len(chunks)])
        if events:
            n_ev += sv.pop_events()[0].shape[0]
        if i >= 30:
            ms.append(t)
    sv.close()
    return {"events": events, "p50_ms": statistics.median(ms), "p99_ms": pct(ms, 0.99), "min_ms": min(ms), "max_ms": max(ms),
            "events_popped": n_ev}


def kernel_arm(dev, nf, iters, reps):
    S = 256
    g = torch.Generator(device=dev).manual_seed(nf)
    walk = torch.cumsum(0.2 * torch.randn((S, nf * iters), device=dev, generator=g), 1).remainder(1.0)   # runs over (0, 1)
    state = torch.zeros((S, 5), dtype=torch.int64, device=dev)
    ev = torch.empty((S, nf + 1, 2), dtype=torch.int64, device=dev)
    counts = torch.empty(S, dtype=torch.int32, device=dev)
    f = b200vad.Binarize(**POLICY).frames(0.01)
    params = _lib.BinarizeParams(f["onset"], f["offset"], f["pad_onset"], f["pad_offset"], f["min_off"], f["min_on"])
    L = b200vad.lib()
    st = torch.cuda.current_stream(dev)
    row = walk.stride(0)

    def run():
        for i in range(iters):
            _lib.check(L.b200vad_regions_step(walk.data_ptr() + 4 * i * nf, S, nf, row, params, state.data_ptr(), None, ev.data_ptr(),
                                              counts.data_ptr(), nf + 1, st.cuda_stream), "b200vad_regions_step")
    run()
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        run()
        e1.record(st)
        e1.synchronize()
        out.append(e0.elapsed_time(e1) * 1000.0 / iters)
    return {"S": S, "nf": nf, "us_per_call_median": statistics.median(out), "us_min": min(out), "us_max": max(out)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pushes", type=int, default=300)
    ap.add_argument("--iters", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    _lib.init(0)
    import oracle
    torch.manual_seed(42)
    o = oracle.VadModel("PyanNet2", {"encoding_dim": 80}).eval()
    blob = b200vad.pack_model(o.model.state_dict(), dev, 80, 4)
    gen = torch.Generator().manual_seed(0)
    chunks = [(0.1 * torch.randn(256, 160, generator=gen)).pin_memory() for _ in range(16)]
    res = {"card": card(), "policy_seconds": POLICY, "push": [], "kernel": []}
    for _ in range(3):
        for events in (False, True):
            r = push_arm(blob, events, chunks, a.pushes)
            res["push"].append(r)
            print(json.dumps(r), flush=True)
    for nf in (1, 500):
        r = kernel_arm(dev, nf, a.iters, a.reps)
        res["kernel"].append(r)
        print(json.dumps(r), flush=True)
    res["card_after"] = card()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
