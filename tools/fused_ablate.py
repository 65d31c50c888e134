"""Timing probes of the fused LSTM layer kernel (csrc/lstm_fused.cu) at the bench shape: per-launch time of the layer kernel
(b200vad_profile_collect kind 0) with parts of the work switched off (b200vad_set_lstm_fused_debug), to see which stage of the
per-step chain MMA -> pointwise -> h exchange -> MMA sets the step time.

    python tools/fused_ablate.py [B T]"""
import ctypes as C
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "universal-voice-activity-detection_b200")):
    sys.path.insert(0, p)

import b200vad  # noqa: E402
import oracle  # noqa: E402


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
    T = int(sys.argv[2]) if len(sys.argv) > 2 else 800
    dev = torch.device("cuda:0")
    lib = b200vad.lib()
    torch.manual_seed(42)
    m = oracle.VadModel("PyanNet2", {"encoding_dim": 80}).eval()
    blob = b200vad.pack_model(m.model.state_dict(), dev, 80, 4)
    x = (torch.randn(B, T, 80, device=dev) * 3 - 5)
    print("clusters:", lib.b200vad_lstm_fused_clusters())

    def run(flags, lag, label, fused=1):
        lib.b200vad_set_lstm_fused(fused)
        lib.b200vad_set_lstm_fused_debug(flags, lag)
        for _ in range(2):
            torch.ops.b200vad.lstm_head(x, blob, 4)
        torch.cuda.synchronize()
        lib.b200vad_profile_enable(1)
        for _ in range(3):
            torch.ops.b200vad.lstm_head(x, blob, 4)
        torch.cuda.synchronize()
        out = []
        for kind in (0, 1):
            ms, n = C.c_double(0), C.c_int(0)
            lib.b200vad_profile_collect(kind, C.byref(ms), C.byref(n))
            out.append((ms.value / max(n.value, 1), n.value))
        lib.b200vad_profile_enable(0)
        print(f"{label:58s} layer kernel {out[0][0]:8.3f} ms x{out[0][1]:3d}   projection {out[1][0]:7.3f} ms x{out[1][1]}", flush=True)

    def waits(flags, label):
        """per-role wait-time table (flag 32): share of the kernel each warp spends in each wait site (non-immediate waits; a
        named barrier counts every passage), and the mbarrier polls (try_wait / test_wait instructions) per step and CTA"""
        lib.b200vad_set_lstm_fused(1)
        lib.b200vad_set_lstm_fused_debug(flags | 32, 3)
        torch.ops.b200vad.lstm_head(x, blob, 4)
        torch.cuda.synchronize()
        W, TAGS, F = 25, 8, 3                                   # warps per CTA, wait tags, fields (cycles, waits, polls): lstm_fused.cu
        n = 148 * W * TAGS * F
        buf = (C.c_longlong * n)()
        lib.b200vad_lstm_fused_read_debug(buf, n)
        roles = {"prod": {1: "x_empty"}, "pw": {6: "acc_ready", 5: "acc_ready bar", 4: "slice bar"}, "mmah": {2: "x_done", 4: "h_ready"},
                 "mmax": {2: "acc_free", 3: "x_full", 5: "drain"}, "send": {1: "slice", 7: "h_free"}}
        role_of = lambda w: "pw" if w < 16 else "prod" if w == 16 else "mmah" if w < 19 else "mmax" if w < 21 else "send"
        at = lambda cta, warp, tag, f: buf[((cta * W + warp) * TAGS + tag) * F + f]
        print(f"--- wait sites, {label} (last layer launch; share of the kernel in non-immediate waits)")
        for cta in (0, 1, 5):
            for warp in (0, 1, 5, 10, 15, 16, 17, 18, 19, 20, 21, 24):
                role = role_of(warp)
                tot = at(cta, warp, 0, 0)
                parts = [f"{roles[role].get(t, t)} {at(cta, warp, t, 0) / max(tot, 1) * 100:5.1f}% (n={at(cta, warp, t, 1)})"
                         for t in range(1, TAGS) if at(cta, warp, t, 1)]
                print(f"cta {cta} warp {warp:2d} {role:5s}: total {tot / 1e6:8.3f} Mcyc  " + "  ".join(parts), flush=True)
        print(f"--- mbarrier polls per step and CTA, {label} (all 25 warps; lane 0 counts the warp's poll instructions)")
        for cta in (0, 1, 5):
            steps = max(at(cta, 16, 0, 1), 1)
            site = {}
            for warp in range(W):
                role = role_of(warp)
                for t in range(1, TAGS):
                    if at(cta, warp, t, 2):
                        k = f"{role}:{roles[role].get(t, t)}"
                        site[k] = site.get(k, 0) + at(cta, warp, t, 2)
            print(f"cta {cta} ({steps} steps): total {sum(site.values()) / steps:7.1f}   " +
                  "  ".join(f"{k} {v / steps:6.1f}" for k, v in sorted(site.items())), flush=True)
        lib.b200vad_set_lstm_fused_debug(0, 3)

    def timeline(flags, label):
        """clock64 stamps of part 0 on CTA 0 over 8 consecutive steps (flag 64), relative to the MMA thread seeing h_ready"""
        lib.b200vad_set_lstm_fused(1)
        lib.b200vad_set_lstm_fused_debug(flags | 64, lag_default)
        torch.ops.b200vad.lstm_head(x, blob, 4)
        torch.cuda.synchronize()
        buf = (C.c_longlong * 128)()
        lib.b200vad_lstm_fused_read_debug(buf, -128)
        names = ["mma:h_ready", "mma:issued", "pw:acc_rdy", "pw:tmem_ld", "pw:ex2", "pw:xchg", "ld:y_done", "pub:slice", "pub:done",
                 "x:start", "pw:math", "ld:issued", "pw:done", "x:xfull", "-", "x:commit"]
        print(f"--- timeline of one part, {label} (cycles after the MMA thread saw h_ready; last column = step period)")
        print("      " + " ".join(f"{n:>12s}" for n in names))
        prev = None
        for st in range(8):
            row = [buf[st * 16 + i] for i in range(len(names))]
            t0 = row[0]
            per = (t0 - prev) if prev is not None else 0
            prev = t0
            print(f"s+{st}: " + " ".join(f"{v - t0:12d}" for v in row) + f"   period {per}", flush=True)
        print("(x:* = the input product of the SAME step and part, issued by the MMA thread one round earlier: negative offsets)")
        lib.b200vad_set_lstm_fused_debug(0, lag_default)

    def mma_threads(label, extra=0):
        """stamps of the two MMA-issuing threads of CTA 0 over two consecutive steps (flag 128)"""
        lib.b200vad_set_lstm_fused(1)
        lib.b200vad_set_lstm_fused_debug(64 | 128 | extra, 2)
        torch.ops.b200vad.lstm_head(x, blob, 4)
        torch.cuda.synchronize()
        buf = (C.c_longlong * 256)()
        lib.b200vad_lstm_fused_read_debug(buf, -256)
        base = 128
        t0 = buf[base]
        print(f"--- MMA threads of CTA 0, {label}: cycles since the recurrent issuer reached (step 100, part 0)")
        for st in range(2):
            for q in range(8):
                h = [buf[base + st * 32 + q * 4 + i] - t0 for i in range(4)]
                xx = [buf[base + 64 + st * 32 + q * 4 + i] - t0 for i in range(4)]
                print(f"step {100 + st} part {q}: H start {h[0]:6d} x_done {h[1]:6d} h_ready {h[2]:6d} committed {h[3]:6d} | "
                      f"X start {xx[0]:6d} acc_free {xx[1]:6d} x_full {xx[2]:6d} committed {xx[3]:6d}", flush=True)
        lib.b200vad_set_lstm_fused_debug(0, 2)

    lag_default = int(os.environ.get("LAG", "2"))
    if os.environ.get("RUNS_ONLY") != "1":
        mma_threads("product path")
        timeline(0, "product path")
        timeline(8 | 16, "no MMAs")
        waits(0, "product path")
        waits(4 | 8 | 16, "no cell math, no MMAs")
    if os.environ.get("RUNS_ONLY") == "3":
        mma_threads("product path")
        mma_threads("no x loads", 256)
        return
    if os.environ.get("RUNS_ONLY") == "2":
        run(0, 2, "fused, product path, prefetch " + os.environ.get("B200VAD_FUSED_PREFETCH", "0"))
        return
    run(0, 2, "legacy (projection + recurrence)", fused=0)
    run(0, 2, "fused, product path")
    run(64, 2, "probe build, all work")
    run(64 | 1, 2, "probe build, HALF the exchange bytes (DSMEM port probe)")
    run(64 | 1 | 8 | 16, 2, "probe build, half exchange, no MMAs")
    run(64 | 256, 2, "probe build, no x loads")
    run(64 | 256 | 1, 2, "probe build, no x loads, half exchange")
    run(64 | 256 | 16, 2, "probe build, no x loads, no input MMAs")
    run(64 | 256 | 8 | 16, 2, "probe build, no x loads, no MMAs")
    run(64 | 256 | 8 | 16 | 1, 2, "probe build, no x loads, no MMAs, half exchange")
    if os.environ.get("RUNS_ONLY") == "1":
        timeline(0, "product path")
        timeline(256, "no x loads")
        timeline(256 | 8 | 16, "no x loads, no MMAs")
        return
    run(4, 2, "no cell math")
    run(8, 2, "no recurrent MMAs")
    run(16, 2, "no input MMAs")
    run(4 | 8 | 16, 2, "no cell math, no MMAs")
    run(8 | 16, 2, "no MMAs at all")
    lib.b200vad_set_lstm_fused_debug(0, 3)


if __name__ == "__main__":
    main()
