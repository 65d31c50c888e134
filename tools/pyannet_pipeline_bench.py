"""PyanNet (SincNet) whole path on one GPU: the one-call op against the current composition, the host session, long-form and
streaming.  Writes one JSON file (default profiles/r03_pyannet_pipeline.json) with the card name and power limit read in the
same run.

  device      4096 x 8 s device-resident: torch.ops.b200vad.vad_pipeline_sincnet against VadModel('PyanNet').predict_step +
              segments(min_run=1), alternated in one process (CUDA events, warm-up), outputs checked equal at that size
  e2e         HostSession(sincnet_packed=...) from pinned f32 and from int16 host waveforms, two slots in flight; the copy-only
              H2D rate of the same bytes gives the PCIe floor (bench.py's h2d_ceiling method)
  longform    1 h recording: reference semantics (5 s windows) and 40500-sample hop
  streaming   256 streams x 5 s window x 270-sample hop: per-push device time p50 / p99

Usage: python tools/pyannet_pipeline_bench.py [--rows 4096] [--seconds 8] [--rounds 5] [--out profiles/r03_pyannet_pipeline.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "universal-voice-activity-detection_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import b200vad  # noqa: E402
from src.engines import VadModel  # noqa: E402

K = 49


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit"], out["max_sm_clock"] = [x.strip() for x in q.split(",")[:2]]
    except Exception as e:  # noqa: BLE001
        out["power_limit"] = f"unread ({e})"
    return out


def events_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def pct(xs, q):
    xs = sorted(xs)
    return xs[min(len(xs) - 1, int(round(q / 100.0 * (len(xs) - 1))))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=4096)
    ap.add_argument("--seconds", type=float, default=8.0)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--chunk-rows", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_pyannet_pipeline.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    dev = torch.device("cuda:0")
    b200vad._lib.init(0)
    res = {"card": card(), "torch": torch.__version__}
    B, N = args.rows, int(args.seconds * 16000)
    Ts = b200vad.host.get_num_frames(N)
    audio_h = B * N / 16000 / 3600
    res["shape"] = {"rows": B, "samples": N, "frames": Ts, "audio_hours_per_step": audio_h}

    torch.manual_seed(42)
    m = VadModel("PyanNet", {}).eval().to(dev)
    with torch.no_grad():   # classifier rescaled so that decisions and segments are not degenerate (random-init logits ~ constant)
        x = m.model(b200vad.synth.meeting_batch(8, N, seed=3).to(dev).unsqueeze(1))
        z = torch.logit(x.clamp(1e-6, 1 - 1e-6))
        scale = 2.0 / z.std().clamp_min(1e-6)
        m.model.classifier.weight.mul_(scale)
        m.model.classifier.bias.copy_((m.model.classifier.bias - z.mean()) * scale)
        m.model.invalidate_packed()
    sd = m.model.state_dict()
    blob = b200vad.pack_model({k: v for k, v in sd.items() if not k.startswith("sincnet.")}, dev, 60, 4)
    sblob = b200vad.pack_sincnet(sd, dev)

    # ---------------- device-resident: new op vs the current composition, alternated
    wav_host = b200vad.synth.meeting_batch(B, N, seed=21)
    wd = wav_host.to(dev)

    def new():
        return torch.ops.b200vad.vad_pipeline_sincnet(wd, blob, sblob, 4, 0.5, K)

    def old():
        with torch.no_grad():
            d = m.predict_step({"inputs": wd}).squeeze(-1).to(torch.uint8)
        return d, torch.ops.b200vad.segments(d, None, 1)

    p_new, d_new, s_new, c_new = new()
    d_old, (s_old, c_old) = old()
    with torch.no_grad():
        p_old = m(wd.unsqueeze(1)).squeeze(-1)
    equal = bool(torch.equal(p_new, p_old) and torch.equal(d_new, d_old) and torch.equal(s_new, s_old) and torch.equal(c_new, c_old))
    del p_new, d_new, s_new, c_new, d_old, s_old, c_old, p_old
    t_new, t_old = [], []
    for _ in range(args.rounds):
        t_old.append(events_ms(old, args.iters))
        t_new.append(events_ms(new, args.iters))
    res["device"] = {"new_op_ms": t_new, "composition_ms": t_old, "new_op_ms_median": pct(t_new, 50),
                     "composition_ms_median": pct(t_old, 50), "new_audio_h_per_s": audio_h / (pct(t_new, 50) / 1e3),
                     "outputs_equal": equal,
                     "note": "median of rounds; each round = iters calls between CUDA events, the two arms alternated; each call "
                             "ends in one blocking read of the segment total"}
    print(json.dumps(res["device"]), flush=True)
    del wd
    torch.cuda.empty_cache()

    # ---------------- end to end through the SincNet host session
    chunk = args.chunk_rows
    sub = B // chunk
    sess = b200vad.HostSession(blob, 4, N, chunk_rows=chunk, sincnet_packed=sblob)
    outs = [dict(), dict()]

    def e2e_run(src, k):
        n = k * sub
        for i in range(n):
            j = i % sub
            if i >= 2:
                sess.wait(i & 1, outs[i & 1])
            sess.submit(i & 1, src[j * chunk:(j + 1) * chunk], 0.5, K, want_dec=True, want_prob=False, out=outs[i & 1])
        for i in range(max(0, n - 2), n):
            sess.wait(i & 1, outs[i & 1])

    e2e = {}
    f32_host = wav_host.pin_memory()
    i16_host = (wav_host * 32768.0).clamp_(-32768, 32767).to(torch.int16).pin_memory()
    for name, src in (("f32", f32_host), ("i16", i16_host)):
        e2e_run(src, 2)
        t0 = time.perf_counter()
        e2e_run(src, args.steps)
        ms = (time.perf_counter() - t0) * 1e3 / args.steps
        e2e[name] = {"ms_per_step": ms, "audio_h_per_s": audio_h / (ms / 1e3), "h2d_bytes_per_step": src.numel() * src.element_size()}
    sess.close()
    probe = torch.empty_like(f32_host, device=dev)
    for _ in range(2):
        probe.copy_(f32_host, non_blocking=True)
    h2d_ms = events_ms(lambda: probe.copy_(f32_host, non_blocking=True), 5)
    e2e["h2d_ceiling_gbs"] = f32_host.numel() * 4 / (h2d_ms / 1e3) / 1e9
    e2e["h2d_floor_ms_per_step_f32"] = h2d_ms
    e2e["note"] = (f"{sub} submissions of {chunk} rows per step, two slots in flight; host wall time over {args.steps} steps after "
                   "2 warm-up steps; h2d ceiling = copy-only rate of the f32 step's bytes")
    res["e2e"] = e2e
    print(json.dumps(e2e), flush=True)
    del probe, f32_host, i16_host, wav_host
    torch.cuda.empty_cache()

    # ---------------- long-form 1 h
    Nl = 3600 * 16000
    g = torch.Generator(device=dev).manual_seed(1)
    wl = 0.05 * torch.randn(Nl, device=dev, generator=g)
    lf = {}
    for name, hop in (("reference_5s_windows", None), ("hop_40500", 40500)):
        v = b200vad.LongFormVad(blob, 4, hop=hop, sincnet_packed=sblob)
        v(wl)
        torch.cuda.synchronize()
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            r = v(wl)
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
        lf[name] = {"ms": pct(ts, 50), "windows": len(r["windows"]), "stream_frames": int(r["stream_dec"].numel()),
                    "audio_h_per_s": 1.0 / (pct(ts, 50) / 1e3)}
    res["longform_1h"] = lf
    print(json.dumps(lf), flush=True)
    del wl
    torch.cuda.empty_cache()

    # ---------------- streaming: 256 streams x 5 s x 270-sample hop
    sv = b200vad.StreamingVad(blob, 4, num_streams=256, window=80000, hop=270, sincnet_packed=sblob)
    gc = torch.Generator().manual_seed(0)
    chunks = [0.1 * torch.randn(256, 270, generator=gc) for _ in range(8)]
    for i in range(5):
        sv.push(chunks[i % 8])
    dev_ms, wall_ms = [], []
    for i in range(100):
        t0 = time.perf_counter()
        _, _, ms = sv.push(chunks[i % 8])
        wall_ms.append((time.perf_counter() - t0) * 1e3)
        dev_ms.append(ms)
    sv.close()
    res["streaming"] = {"streams": 256, "window": 80000, "hop": 270, "pushes": 100,
                        "device_ms_p50": pct(dev_ms, 50), "device_ms_p99": pct(dev_ms, 99),
                        "wall_ms_p50": pct(wall_ms, 50), "wall_ms_p99": pct(wall_ms, 99),
                        "note": "CUDA graph replay per push, chunks from pageable host tensors"}
    print(json.dumps(res["streaming"]), flush=True)

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
