"""bench.py's command line and its --dump-outputs writer, on the host (the GPU run is bench.py itself)."""
import os
import subprocess
import sys

import numpy as np
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _dir_bytes(d):
    return sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))


def test_dump_outputs_types_budget_and_sample(tmp_path):
    g = torch.Generator().manual_seed(0)
    prob = torch.rand(4096, 800, generator=g)
    dec = (prob > 0.5).to(torch.uint8)
    counts = torch.randint(0, 300, (4096,), dtype=torch.int32, generator=g)
    segs = torch.randint(0, 1 << 22, (1_500_000, 3), dtype=torch.int32, generator=g)      # more than its share of the budget
    out = {"prob": prob, "dec": dec, "counts": counts, "segments": segs}
    bench.dump_outputs(str(tmp_path), out)
    assert sorted(os.listdir(tmp_path)) == ["counts.npy", "dec.npy", "prob.npy", "segments.npy", "segments_rows.npy"]
    assert _dir_bytes(tmp_path) <= bench.DUMP_BYTES
    z = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert z["prob"].dtype == np.float32 and np.array_equal(z["prob"], prob.numpy())
    assert z["dec"].dtype == np.float32 and np.array_equal(z["dec"], dec.numpy())
    assert z["counts"].dtype == np.float64 and np.array_equal(z["counts"], counts.numpy())
    idx = z["segments_rows"].astype(np.int64)
    assert z["segments"].dtype == np.float64 and len(idx) > 100_000 and np.all(np.diff(idx) > 0)
    assert np.array_equal(z["segments"], segs.numpy()[idx])
    # the sample is fixed: a second dump writes the same rows
    bench.dump_outputs(str(tmp_path / "again"), out)
    assert np.array_equal(np.load(tmp_path / "again" / "segments_rows.npy"), z["segments_rows"])
    # a dump into the same directory whose arrays fit leaves no stale sample index behind
    bench.dump_outputs(str(tmp_path), {"segments": segs[:10]})
    assert not os.path.exists(tmp_path / "segments_rows.npy")


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--steps" in r.stderr
