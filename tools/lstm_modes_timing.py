"""Per-launch time of the LSTM layer kernels at the bench shape for the three layer modes (b200vad_set_lstm_fused: 2 = fused on
CTA pairs, 1 = fused, 0 = projection GEMM + recurrence), CUDA events inside the library (b200vad_profile_collect).

    python tools/lstm_modes_timing.py [B T] [modes, e.g. 21]

B may be a comma-separated list: the step time by parts in flight of the launcher's table (kStepUs in csrc/lstm_fused.cu) is
`python tools/lstm_modes_timing.py 256,512,768,1024,1280,1536,1792,2048 500 1` (one wave of n = B / 256 parts per cluster on
the 33 clusters of a B200; us per step = layer kernel ms / T x 1000)."""
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
    Bs = [int(b) for b in sys.argv[1].split(",")] if len(sys.argv) > 1 else [4096]
    T = int(sys.argv[2]) if len(sys.argv) > 2 else 800
    # a mode may carry the pair-kernel tuning bits as a suffix: "2.0" = mode 2 with b200vad_set_lstm_pair_opt(0)
    modes = (sys.argv[3] if len(sys.argv) > 3 else "2,1,0").split(",")
    dev = torch.device("cuda:0")
    lib = b200vad.lib()
    torch.manual_seed(42)
    m = oracle.VadModel("PyanNet2", {"encoding_dim": 80}).eval()
    blob = b200vad.pack_model(m.model.state_dict(), dev, 80, 4)
    for B in Bs:
        if len(Bs) > 1:
            print(f"B = {B}, T = {T}", flush=True)
        run(lib, blob, torch.randn(B, T, 80, device=dev) * 3 - 5, modes)
    lib.b200vad_set_lstm_fused(1)


def run(lib, blob, x, modes):
    ref = None
    for mspec in modes:
        mode = int(mspec.split(".")[0])
        if "." in mspec:
            lib.b200vad_set_lstm_pair_opt(int(mspec.split(".")[1]))
        lib.b200vad_set_lstm_fused(mode)
        for _ in range(2):
            p = torch.ops.b200vad.lstm_head(x, blob, 4)
        torch.cuda.synchronize()
        lib.b200vad_profile_enable(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            p = torch.ops.b200vad.lstm_head(x, blob, 4)
        e1.record()
        torch.cuda.synchronize()
        out = []
        for kind in (0, 1):
            ms, n = C.c_double(0), C.c_int(0)
            lib.b200vad_profile_collect(kind, C.byref(ms), C.byref(n))
            out.append((ms.value / max(n.value, 1), n.value))
        lib.b200vad_profile_enable(0)
        if ref is None:
            ref = p.clone()
        diff = (p - ref).abs().max().item()
        print(f"mode {mspec}: layer kernel {out[0][0]:7.3f} ms x{out[0][1]}  projection {out[1][0]:7.3f} ms x{out[1][1]}  "
              f"lstm_head {e0.elapsed_time(e1) / 5:7.3f} ms  max |p - p(first mode)| {diff:.3e}", flush=True)


if __name__ == "__main__":
    main()
