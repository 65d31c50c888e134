"""Exact tests of the integer kernels either side of the model over their whole parameter range: threshold + median
filter, run-length segments and their output cap (C ABI, device pipeline, host session), interval scoring, stat scores,
long-form stitching and the streaming ring buffer.  These kernels have no tolerance to hide behind, so every output is
compared with torch.equal against a plain CPU reference written here, at the tile, halo, chunk, word and grid-split edges
where such kernels go wrong."""
import ctypes as C
import warnings

import numpy as np
import pytest
import torch
from scipy.signal import medfilt

import util

pytestmark = pytest.mark.gpu

EINVAL = -1          # B200VAD_EINVAL
TILE = 2048          # frames per CTA of the median kernel
CHUNK = 256          # frames per iteration of the segments kernel
K = 5                # median window of the pipeline / session tests: short, so that rows hold several segments


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import b200vad
    b200vad._lib.init(0)
    return torch.device("cuda:0")


def _lib():
    import b200vad
    return b200vad.lib()


def _st(dev):
    return torch.cuda.current_stream(dev).cuda_stream


# ---------------------------------------------------------------- threshold + median
def _median_ref(p: np.ndarray, thr: float, k: int) -> np.ndarray:
    """oracle.median_filter with an explicit window: torch.where(p < thr, 0, 1), then scipy's zero-padded medfilt per row"""
    d = np.where(p < np.float32(thr), 0, 1).astype(np.int64)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")          # a window longer than the row: medfilt warns, then zero pads as usual
        return medfilt(d, [1, k]).astype(np.int64)


def _blocks(g, T, lens):
    """0/1 row made of alternating runs whose lengths are drawn from lens"""
    ends = np.cumsum(g.choice(lens, T))                          # T runs of >= 1 frame cover the row
    run = np.searchsorted(ends, np.arange(T), side="right")       # index of the run each frame is in
    return (run + g.integers(2)) % 2 == 1


def _median_rows(T, thr, k, seed):
    """(5, T) float32 rows: a random walk around thr, uniform noise, runs whose lengths sit at the median's vote count
    ((k+1)/2 of k) made of thr itself and the float just below it, the same runs made of NaN / +-inf / thr, and values at
    log-spread distances from thr"""
    g = np.random.default_rng(seed)
    t = np.float32(thr)
    below = np.nextafter(t, np.float32(-np.inf))
    half = k // 2
    lens = [n for n in (1, half, half + 1, half + 2, k - 1, k, k + 1) if n >= 1]
    hi = np.array([np.nan, np.inf, t] + ([0.0, -0.0] if t == 0 else []), np.float32)
    lo = np.array([-np.inf, below], np.float32)
    rows = np.empty((5, T), np.float32)
    rows[0] = t + 0.3 * np.cumsum(g.standard_normal(T))
    rows[1] = t + g.uniform(-1, 1, T)
    rows[2] = np.where(_blocks(g, T, lens), t, below)
    rows[3] = np.where(_blocks(g, T, lens), g.choice(hi, T), g.choice(lo, T))
    rows[4] = t + g.choice([-1.0, 1.0], T) * 10.0 ** g.uniform(-5, 0, T)
    return rows


MEDIAN_K = list(range(1, 62, 2)) + [1023, 1025]
THRESHOLDS = [0.5, 0.0, -0.0, 1.0, 0.3]


@pytest.mark.parametrize("k", MEDIAN_K)
def test_threshold_median_every_window(dev, k):
    """every odd k to 61 and the largest two: rows of one frame, around k, and around one, two and three 2048-frame tiles
    (where the window's halo reaches into the neighbouring tile), at each threshold, for both output types"""
    Ts = sorted({1, k - 1, k, TILE - 1, TILE, TILE + 1, 2 * TILE + k // 2, 3 * TILE + 1} - {0})
    for T in Ts:
        for i, thr in enumerate(THRESHOLDS):
            p = _median_rows(T, thr, k, seed=1000 * k + 10 * T + i)
            want = torch.from_numpy(_median_ref(p, thr, k))
            x = torch.from_numpy(p).to(dev)
            for as_int64 in (False, True):
                got = torch.ops.b200vad.threshold_median(x, thr, k, as_int64)
                assert got.dtype == (torch.int64 if as_int64 else torch.uint8)
                assert torch.equal(got.cpu().long(), want), (T, thr, as_int64)


def test_threshold_median_refuses_bad_windows(dev):
    import b200vad
    L = _lib()
    x = torch.rand(2, 100, device=dev)
    out = torch.zeros(2, 100, dtype=torch.uint8, device=dev)
    for k in (1027, 2049, 0, 2, 48, 1024, -1):
        assert L.b200vad_threshold_median(x.data_ptr(), 2, 100, 0.5, k, out.data_ptr(), 1, None, 0.0, _st(dev)) == EINVAL, k
        with pytest.raises(b200vad.B200VadError):
            torch.ops.b200vad.threshold_median(x, 0.5, k, False)
    torch.cuda.synchronize()
    assert not out.any()                                 # nothing was launched


@pytest.mark.parametrize("k", [1, 49, 1025])
def test_threshold_median_near_count(dev, k):
    """near_count of b200vad_threshold_median (C ABI) is ((p - thr).abs() <= tol).sum() over the whole batch: frames near a
    tile edge are also read as the next tile's halo and must still count once"""
    L = _lib()
    for T in (1, TILE - 1, TILE, TILE + 1, 2 * TILE + k // 2, 3 * TILE + 1):
        for thr in (0.5, 0.0, 0.3):
            for tol in (0.0, 1e-3, 0.25):
                p = _median_rows(T, thr, k, seed=T + k)
                x = torch.from_numpy(p).to(dev)
                out = torch.empty(p.shape, dtype=torch.uint8, device=dev)
                near = torch.zeros(1, dtype=torch.int32, device=dev)
                rc = L.b200vad_threshold_median(x.data_ptr(), p.shape[0], T, thr, k, out.data_ptr(), 1, near.data_ptr(), tol, _st(dev))
                assert rc == 0
                xc = torch.from_numpy(p)
                assert int(near.item()) == int(((xc - thr).abs() <= tol).sum()), (T, thr, tol)
                assert torch.equal(out.cpu().long(), torch.from_numpy(_median_ref(p, thr, k)))


def test_threshold_median_splits_large_batches(dev):
    """more than 32768 rows: the op cuts the batch into several C calls"""
    B, T, k = 32769, 37, 5
    g = np.random.default_rng(7)
    p = g.random((B, T), dtype=np.float32)
    want = torch.from_numpy(_median_ref(p, 0.5, k))
    x = torch.from_numpy(p).to(dev)
    for as_int64 in (False, True):
        assert torch.equal(torch.ops.b200vad.threshold_median(x, 0.5, k, as_int64).cpu().long(), want)


# ---------------------------------------------------------------- run-length segments
def _runs(row, min_run):
    """(first, last) of every run of non-zero frames that is at least min_run frames long"""
    a = np.asarray(row) != 0
    d = np.diff(np.concatenate([[0], a.astype(np.int8), [0]]))
    s, e = np.nonzero(d == 1)[0], np.nonzero(d == -1)[0] - 1
    keep = e - s + 1 >= min_run
    return list(zip(s[keep].tolist(), e[keep].tolist()))


def _seg_ref(streams, min_run):
    """(S, 3) int32 (stream, first, last) ordered by (stream, first), and the per-stream counts"""
    rows = [(r, a, b) for r, s in enumerate(streams) for a, b in _runs(s, min_run)]
    counts = torch.tensor([len(_runs(s, min_run)) for s in streams], dtype=torch.int32)
    return torch.tensor(rows, dtype=torch.int32).reshape(-1, 3), counts


def _segment_rows(T, seed):
    """(R, T) uint8 decisions: random densities, non-zero bytes other than 1, runs that start or end exactly on the
    kernel's 256-frame chunk edges, runs that span three or more chunks, runs of every length around the min_run values"""
    g = np.random.default_rng(seed)
    rows = []
    for dens in (0.1, 0.5, 0.9):
        rows.append((g.random(T) < dens).astype(np.uint8))
    rows.append(np.where(g.random(T) < 0.6, g.integers(1, 256, T), 0).astype(np.uint8))
    edges = np.zeros(T, np.uint8)
    for a, b in ((0, CHUNK - 1), (CHUNK, 2 * CHUNK - 1), (2 * CHUNK - 1, 2 * CHUNK), (3 * CHUNK - 2, 3 * CHUNK - 1),
                 (3 * CHUNK + 1, 4 * CHUNK)):
        edges[a:b + 1] = 1
    rows.append(edges)
    for a, b in ((CHUNK, 4 * CHUNK + 10), (100, 900), (CHUNK - 1, 3 * CHUNK), (0, 3 * CHUNK - 1)):
        r = np.zeros(T, np.uint8)
        r[a:b + 1] = 1
        rows.append(r)
    lens = list(range(1, 10)) + [CHUNK - 1, CHUNK, CHUNK + 1, 299, 300, 301]
    ladder, pos = np.zeros(T, np.uint8), 3
    for n in g.permutation(lens * 3):
        ladder[pos:pos + n] = 1
        pos += int(n) + 1 + int(g.integers(0, 3))
    rows.append(ladder)
    rows.append(np.ones(T, np.uint8))
    rows.append(np.zeros(T, np.uint8))
    rows.append((np.arange(T) % 2).astype(np.uint8))
    return np.stack(rows)[:, :T]


@pytest.mark.parametrize("min_run", [1, 2, 3, 7, 300])
def test_segments_chunk_edges(dev, min_run):
    import oracle
    for T in (1, 2, CHUNK - 1, CHUNK, CHUNK + 1, 3 * CHUNK, 5 * CHUNK + 3, 8 * CHUNK - 1):
        d = _segment_rows(T, seed=T)
        if min_run == 2:                                     # the helper is the pinned oracle's RLE at the fbank path's min_run
            assert all(_runs(r, 2) == oracle.postproc.rle_frames(r) for r in d)
        want, counts = _seg_ref(d, min_run)
        seg, c = torch.ops.b200vad.segments(torch.from_numpy(d).to(dev), None, min_run)
        assert torch.equal(seg.cpu(), want), T
        assert torch.equal(c.cpu(), counts), T


def _ragged_streams(seed):
    """empty and one-frame streams, all-ones streams of 256 m - 1, 256 m and 256 m + 1 frames, random streams"""
    g = np.random.default_rng(seed)
    streams = [np.zeros(0, np.uint8), np.ones(1, np.uint8), np.zeros(1, np.uint8), np.zeros(0, np.uint8)]
    for m in (1, 2, 3, 5):
        for n in (CHUNK * m - 1, CHUNK * m, CHUNK * m + 1):
            streams.append(np.ones(n, np.uint8))
    streams.append(np.ones(1, np.uint8))
    for n in g.integers(0, 1500, 12):
        streams.append((g.random(n) < g.random()).astype(np.uint8))
    streams.append(np.zeros(0, np.uint8))
    return streams


@pytest.mark.parametrize("min_run", [1, 2, 3, 7, 300])
def test_segments_offsets_path(dev, min_run):
    streams = _ragged_streams(seed=min_run)
    flat = torch.from_numpy(np.concatenate(streams))
    offsets = torch.tensor(np.concatenate([[0], np.cumsum([len(s) for s in streams])]), dtype=torch.int64)
    want, counts = _seg_ref(streams, min_run)
    seg, c = torch.ops.b200vad.segments(flat.to(dev), offsets.to(dev), min_run)
    assert torch.equal(seg.cpu(), want) and torch.equal(c.cpu(), counts)


def _segments_c(dev, d, offsets, R, T, min_run, cap, rows):
    """b200vad_segments into buffers pre-filled with -7; returns (seg, counts, seg_off) on the host"""
    L = _lib()
    seg = torch.full((rows, 3), -7, dtype=torch.int32, device=dev)
    counts = torch.full((R,), -7, dtype=torch.int32, device=dev)
    seg_off = torch.full((R + 1,), -7, dtype=torch.int64, device=dev)
    rc = L.b200vad_segments(d.data_ptr(), None if offsets is None else offsets.data_ptr(), R, T, min_run, counts.data_ptr(),
                            seg_off.data_ptr(), seg.data_ptr(), cap, _st(dev))
    assert rc == 0
    return seg.cpu(), counts.cpu(), seg_off.cpu()


@pytest.mark.parametrize("min_run", [1, 2])
def test_segments_cap_truncates(dev, min_run):
    """b200vad_segments with cap below the total writes exactly the first cap entries of the full (row, start)-ordered list
    and nothing after them; counts and seg_off still describe the full list"""
    T = 5 * CHUNK + 3
    d = _segment_rows(T, seed=11)
    streams = _ragged_streams(seed=12)
    flat = np.concatenate(streams)
    offsets = torch.tensor(np.concatenate([[0], np.cumsum([len(s) for s in streams])]), dtype=torch.int64)
    for name, rows_in, buf, offs, T_arg in (("uniform", list(d), torch.from_numpy(d), None, T),
                                            ("offsets", streams, torch.from_numpy(flat), offsets, 0)):
        want, counts = _seg_ref(rows_in, min_run)
        R, total = len(rows_in), want.shape[0]
        assert total >= 3
        seg_off = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(counts.long(), 0)])
        x = buf.to(dev)
        o = None if offs is None else offs.to(dev)
        for cap in sorted({0, 1, total // 2, total - 1, total}):
            seg, c, so = _segments_c(dev, x, o, R, T_arg, min_run, cap, total + 4)
            assert torch.equal(seg[:cap], want[:cap]), (name, cap)
            assert bool((seg[cap:] == -7).all()), (name, cap)
            assert torch.equal(c, counts) and torch.equal(so, seg_off), (name, cap)


@pytest.fixture(scope="module")
def fbank_model(dev):
    """PyanNet2 with a spread head, 12 two-second rows, and the median of their probabilities as the threshold (so that
    about half the frames are speech and the rows hold several segments)"""
    import b200vad
    wav = util.synth_wave(12, 32000, seed=5)
    feats = torch.ops.b200vad.fbank(wav.to(dev), None).cpu()
    o = util.make_oracle("PyanNet2", {"encoding_dim": 80}, spread=True, feats=feats)
    blob = b200vad.pack_model(o.model.state_dict(), dev, 80, 4)
    prob, _, _, _ = torch.ops.b200vad.vad_pipeline(wav.to(dev), None, blob, 4, 0.5, K)
    return wav, blob, float(prob.median())


def _full_pipeline(dev, wav, blob, thr):
    prob, dec, seg, counts = torch.ops.b200vad.vad_pipeline(wav.to(dev), None, blob, 4, thr, K)
    want, want_counts = _seg_ref(list(dec.cpu().numpy()), 2)
    assert torch.equal(seg.cpu(), want) and torch.equal(counts.cpu(), want_counts)
    print(f"{want.shape[0]} segments in {wav.shape[0]} rows")
    assert want.shape[0] >= 4
    return prob.cpu(), dec.cpu(), want, want_counts


def test_pipeline_segment_cap(dev, fbank_model):
    """b200vad_pipeline_fbank_f32 with a segment cap below the total: the first cap segments of the full list, nothing after
    them, and unchanged probabilities, decisions, counts and offsets"""
    wav, blob, thr = fbank_model
    prob, dec, want, counts = _full_pipeline(dev, wav, blob, thr)
    L = _lib()
    B, N = wav.shape
    total = want.shape[0]
    x = wav.to(dev)
    ws = torch.empty(L.b200vad_pipeline_workspace_bytes(B, N), dtype=torch.uint8, device=dev)
    for cap in (0, 1, total // 2, total - 1):
        p = torch.empty(prob.shape, device=dev)
        d = torch.empty(dec.shape, dtype=torch.uint8, device=dev)
        c = torch.full((B,), -7, dtype=torch.int32, device=dev)
        so = torch.full((B + 1,), -7, dtype=torch.int64, device=dev)
        seg = torch.full((total + 4, 3), -7, dtype=torch.int32, device=dev)
        rc = L.b200vad_pipeline_fbank_f32(blob.data_ptr(), 4, x.data_ptr(), None, B, N, N, thr, K, p.data_ptr(), d.data_ptr(),
                                          c.data_ptr(), so.data_ptr(), seg.data_ptr(), cap, ws.data_ptr(), ws.numel(), _st(dev))
        assert rc == 0
        seg = seg.cpu()
        assert torch.equal(seg[:cap], want[:cap]) and bool((seg[cap:] == -7).all()), cap
        assert torch.equal(p.cpu(), prob) and torch.equal(d.cpu(), dec) and torch.equal(c.cpu(), counts)
        assert so.cpu().tolist() == [0] + torch.cumsum(counts.long(), 0).tolist()


def test_host_session_segment_cap(dev, fbank_model):
    """b200vad_session_run_host over four chunks of 3 rows with caps on, either side of and between the chunks' segment
    boundaries: the host buffer holds the first cap segments of the full list and nothing after them, and the reported
    number is the full total"""
    import b200vad
    wav, blob, thr = fbank_model
    _, _, want, _ = _full_pipeline(dev, wav, blob, thr)
    B, N = wav.shape
    total = want.shape[0]
    sess = b200vad.HostSession(blob, 4, N, chunk_rows=3)
    src = wav.pin_memory()
    assert torch.equal(sess.run(src, thr, K)["seg"], want)
    cuts = [int((want[:, 0] < r).sum()) for r in (3, 6, 9)]
    caps = {0, 1, total - 1, total, total + 3}
    for cut in cuts:
        caps |= {cut - 1, cut, cut + 1}
    L = _lib()
    for cap in sorted(c for c in caps if 0 <= c <= total + 3):
        buf = torch.full((total + 4, 3), -7, dtype=torch.int32).pin_memory()
        nseg = C.c_int64(-1)
        rc = L.b200vad_session_run_host(sess._h, src.data_ptr(), B, thr, K, None, None, buf.data_ptr(), cap, C.byref(nseg))
        assert rc == 0 and nseg.value == total, cap
        n = min(cap, total)
        assert torch.equal(buf[:n], want[:n]) and bool((buf[n:] == -7).all()), cap
    sess.close()


# ---------------------------------------------------------------- interval scoring
def _score_ref(gt, pred, nframes):
    """fa / md frames per recording: get_binary_tensor's t[start:end] = 1 with Python's slice clamping of negative,
    reversed and past-the-end bounds (predict.py:660), then the logical ands of predict.py:666-673"""
    off = np.concatenate([[0], np.cumsum(nframes)]).astype(np.int64)
    masks = []
    for iv in (gt, pred):
        flat = np.zeros(int(off[-1]), bool)
        for r, s, e in iv.tolist():
            flat[off[r]:off[r + 1]][s:e] = True
        masks.append(flat)
    g, p = masks
    cfa = np.concatenate([[0], np.cumsum(p & ~g)])
    cmd = np.concatenate([[0], np.cumsum(g & ~p)])
    return torch.from_numpy(cfa[off[1:]] - cfa[off[:-1]]), torch.from_numpy(cmd[off[1:]] - cmd[off[:-1]])


def _score(dev, gt, pred, nframes):
    words = (nframes.astype(np.int64) + 31) // 32
    word_off = np.concatenate([[0], np.cumsum(words)])
    fa, md = torch.ops.b200vad.score_intervals(torch.from_numpy(gt).to(dev), torch.from_numpy(pred).to(dev),
                                               torch.from_numpy(word_off).to(dev), torch.from_numpy(nframes).to(dev),
                                               int(word_off[-1]), int(words.max()))
    return fa.cpu(), md.cpu()


def _iv(rows):
    return np.asarray(rows, dtype=np.int32).reshape(-1, 3)


def test_score_intervals_every_word_bit(dev):
    """one recording of 97 frames per (start, end) pair, both from -3 to 99: negative, reversed, empty and past-the-end
    bounds, and every start and end bit of the four 32-frame words; the prediction of each recording is another pair"""
    nf = 97
    pairs = [(s, e) for s in range(-3, nf + 3) for e in range(-3, nf + 3)]
    perm = np.random.default_rng(1).permutation(len(pairs))
    gt = _iv([(r, s, e) for r, (s, e) in enumerate(pairs)])
    pred = _iv([(r, *pairs[perm[r]]) for r in range(len(pairs))])
    nframes = np.full(len(pairs), nf, np.int32)
    fa, md = _score(dev, gt, pred, nframes)
    want_fa, want_md = _score_ref(gt, pred, nframes)
    assert torch.equal(fa, want_fa) and torch.equal(md, want_md)


def test_score_intervals_bounds_and_overlaps(dev):
    """frame counts that are not multiples of 32 (and 0), recordings without intervals, int32 extremes, overlapping and
    duplicate intervals listed in no particular order"""
    g = np.random.default_rng(2)
    I32 = np.iinfo(np.int32)
    nframes = np.array([0, 1, 31, 32, 33, 63, 64, 65, 100, 1000, 4097, 77, 5, 4096], np.int32)
    R = len(nframes)
    rows = {"gt": [], "pred": []}
    for r, nf in enumerate(nframes.tolist()):
        edge = [I32.min, -nf - 5, -nf, -nf + 1, -33, -32, -31, -1, 0, 1, 31, 32, 33, 63, 64, 65, nf - 1, nf, nf + 1, I32.max]
        for key in rows:
            if r == R - 1 and key == "pred":
                continue                                         # a recording with ground truth only
            for _ in range(int(g.integers(0, 12))):
                rows[key].append((r, int(g.choice(edge)), int(g.choice(edge))))
            for _ in range(int(g.integers(0, 6))):
                a = int(g.integers(-nf - 3, nf + 3)) if nf else 0
                rows[key].append((r, a, a + int(g.integers(0, 70))))
    for key in rows:
        rows[key] += rows[key][::3]                              # duplicates
        rows[key] = [rows[key][i] for i in g.permutation(len(rows[key]))]
    gt, pred = _iv(rows["gt"]), _iv(rows["pred"])
    fa, md = _score(dev, gt, pred, nframes)
    want_fa, want_md = _score_ref(gt, pred, nframes)
    assert torch.equal(fa, want_fa) and torch.equal(md, want_md)
    assert int(want_fa.sum()) > 0 and int(want_md.sum()) > 0
    # no prediction at all / no interval at all
    fa, md = _score(dev, gt, _iv([]), nframes)
    assert torch.equal(fa, torch.zeros(R, dtype=torch.int64)) and torch.equal(md, _score_ref(gt, _iv([]), nframes)[1])
    fa, md = _score(dev, _iv([]), _iv([]), nframes)
    assert not fa.any() and not md.any()


def test_score_intervals_past_the_grid_split(dev):
    """70 000 short recordings: the per-recording count kernel runs as two launches of at most 65 535 recordings"""
    g = np.random.default_rng(3)
    R = 70000
    nframes = g.integers(0, 130, R).astype(np.int32)
    rows = {}
    for key in ("gt", "pred"):
        n = g.integers(0, 4, R)
        r = np.repeat(np.arange(R), n)
        nf = nframes[r].astype(np.int64)
        s = np.floor(g.random(r.size) * (nf + 20)).astype(np.int64) - 10
        e = s + g.integers(-5, 60, r.size)
        rows[key] = np.stack([r, s, e], 1).astype(np.int32)
    gt, pred = rows["gt"], rows["pred"]
    fa, md = _score(dev, gt, pred, nframes)
    want_fa, want_md = _score_ref(gt, pred, nframes)
    assert torch.equal(fa, want_fa) and torch.equal(md, want_md)
    assert int(want_fa[65535:].sum()) > 0 and int(want_md[65535:].sum()) > 0


# ---------------------------------------------------------------- stat scores
def test_stat_scores_unaligned_views(dev):
    """decisions and labels at byte offsets 0-15 (the kernel reads 16-byte vectors only when both are aligned), lengths
    around multiples of 16, and non-zero bytes other than 1"""
    g = torch.Generator().manual_seed(3)
    n_max = 65537
    bytes_of = lambda: torch.where(torch.rand(n_max + 16, generator=g) < 0.5, 0,
                                   torch.randint(1, 256, (n_max + 16,), generator=g)).to(torch.uint8)
    dh, lh = bytes_of(), bytes_of()
    dd, ld = dh.to(dev), lh.to(dev)
    for n in (1, 15, 16, 17, 31, 32, 33, 255, 256, 257, 4095, 4096, 4097, 65535, 65536, 65537):
        for od in range(16):
            for ol in sorted({od, 0, (7 * od + 3) % 16}):
                got = torch.ops.b200vad.stat_scores(dd[od:od + n], ld[ol:ol + n]).cpu()
                d, y = dh[od:od + n] != 0, lh[ol:ol + n] != 0
                want = torch.stack([(d & y).sum(), (d & ~y).sum(), (~d & ~y).sum(), (~d & y).sum()])
                assert torch.equal(got, want), (n, od, ol)


# ---------------------------------------------------------------- long-form stitching
@pytest.mark.parametrize("W", [1, 2, 7])
@pytest.mark.parametrize("Tw", [1, 2, 9, 10, 500])
def test_stitch_center(dev, W, Tw):
    """hop 1, Tw - 1 and Tw (odd and even Tw - hop), stream lengths below, at and past the last window, where the stream is
    filled with 0"""
    from oracle import longform as olf
    prob = (torch.arange(W * Tw, dtype=torch.float32) + 1).reshape(W, Tw)       # every (window, frame) distinct and non-zero
    x = prob.to(dev)
    for hop in sorted({1, Tw - 1, Tw} - {0}):
        end = W * hop + Tw
        for L in sorted({0, 1, (W - 1) * hop + Tw, end - 1, end, end + 1, end + 37}):
            got = torch.ops.b200vad.stitch_center(x, hop, L).cpu()
            assert torch.equal(got, torch.from_numpy(olf.stitch_center(prob.numpy(), hop, L))), (hop, L)


def test_stitch_center_refuses_bad_hops(dev):
    L = _lib()
    x = torch.ones(3, 10, device=dev)
    out = torch.empty(40, device=dev)
    for hop in (0, -1, 11):
        assert L.b200vad_stitch_center(x.data_ptr(), 3, 10, hop, out.data_ptr(), 40, _st(dev)) == EINVAL, hop


# ---------------------------------------------------------------- streaming ring buffer
@pytest.fixture(scope="module")
def stream_models(dev):
    """random-init fbank -> PyanNet2 blob and SincNet -> PyanNet blobs (only the buffered windows are checked here)"""
    import b200vad
    o2 = util.make_oracle("PyanNet2", {"encoding_dim": 80})
    o1 = util.make_oracle("PyanNet", {})
    sd = o1.model.state_dict()
    return {"fbank": (b200vad.pack_model(o2.model.state_dict(), dev, 80, 4), None),
            "sincnet": (b200vad.pack_model({k: v for k, v in sd.items() if not k.startswith("sincnet.")}, dev, 60, 4),
                        b200vad.pack_sincnet(sd, dev))}


@pytest.mark.parametrize("front,S,window,hop,graph", [("fbank", 3, 1600, 480, True), ("fbank", 2, 800, 800, False),
                                                      ("sincnet", 3, 2000, 270, True), ("sincnet", 2, 1999, 540, False)])
def test_stream_ring_wraps(dev, stream_models, front, S, window, hop, graph):
    """hops that do not divide the window (or equal it), the ring wrapped at least 5 times: after every push the buffered
    window is the last `window` samples of the stream (zeros before the first sample), and the push returns the newest
    frames of that window"""
    import b200vad
    blob, sblob = stream_models[front]
    sv = b200vad.StreamingVad(blob, 4, num_streams=S, window=window, hop=hop, use_graph=graph, sincnet_packed=sblob)
    g = torch.Generator().manual_seed(window + hop)
    model = np.zeros((S, window), np.float32)
    pushes = 5 * window // hop + 3
    for i in range(pushes):
        chunk = 0.1 * torch.randn(S, hop, generator=g)
        prob, dec, _ = sv.push(chunk if i % 2 else chunk.to(dev))
        model = np.concatenate([model, chunk.numpy()], 1)[:, -window:]
        w, p_all, d_all = sv.snapshot()
        assert torch.equal(w, torch.from_numpy(model)), i
        assert torch.equal(prob, p_all[:, -sv.nf:]) and torch.equal(dec, d_all[:, -sv.nf:]), i
    sv.close()
