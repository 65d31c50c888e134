"""GPU tests of LongFormVad over many recordings at once: every recording of a list call equals its own single call bit for bit
(both front ends, hop = window and overlapped, threshold / median and Binarize), across launch boundaries, from int16 input and
from views of one buffer fenced by NaN samples; the ragged stitching and smoothing kernels against the oracle; one full-size
call."""
import numpy as np
import pytest
import torch

import util

pytestmark = pytest.mark.gpu

# 2 s (no window under reference semantics), exactly one window, a kept 3.9 s tail, a dropped 2 s tail, shorter than one
# window, SincNet's 991-sample minimum, 10 min
LENGTHS = [32000, 80000, 302400, 272000, 20000, 991, 9_600_000]
POLICY = dict(onset=0.6, offset=0.4, min_duration_on=0.2, min_duration_off=0.3, pad_onset=0.05, pad_offset=0.1)


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import b200vad
    b200vad._lib.init(0)
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def models(dev):
    """{'fbank': (blob, None), 'sincnet': (blob, sincnet blob)} with probabilities spread over (0, 1)"""
    import b200vad
    import oracle
    wav = util.synth_wave(4, 80000, seed=5)
    o = util.make_oracle("PyanNet2", {"encoding_dim": 80}, spread=True, feats=oracle.lhotse_fbank(wav), sigma=2.0)
    fb = b200vad.pack_model(o.model.state_dict(), dev, 80, 4)
    o = util.make_oracle("PyanNet", {}, spread=True, feats=wav, sigma=2.0)
    sd = o.model.state_dict()
    sb = b200vad.pack_model({k: v for k, v in sd.items() if not k.startswith("sincnet.")}, dev, 60, 4)
    return {"fbank": (fb, None), "sincnet": (sb, b200vad.pack_sincnet(sd, dev))}


def _recordings(lengths, seed):
    return [util.synth_wave(1, n, seed=seed + i)[0] if n else torch.zeros(0) for i, n in enumerate(lengths)]


def _lf(models, front, hop, binarize, max_rows=4096):
    import b200vad
    blob, sblob = models[front]
    if hop is not None:
        hop = 270 * 120 if sblob is not None else 40000
    return b200vad.LongFormVad(blob, 4, hop=hop, sincnet_packed=sblob, max_rows=max_rows,
                               binarize=b200vad.Binarize(**POLICY) if binarize else None)


def _same(a, b):
    assert a["windows"] == b["windows"]
    assert a["prob"].shape == b["prob"].shape and torch.equal(a["prob"], b["prob"])
    assert a["stream_dec"].dtype == b["stream_dec"].dtype and torch.equal(a["stream_dec"], b["stream_dec"])
    assert a["intervals"] == b["intervals"]


@pytest.mark.parametrize("binarize", [False, True])
@pytest.mark.parametrize("hop", [None, "overlap"])
@pytest.mark.parametrize("front", ["fbank", "sincnet"])
def test_each_recording_equals_its_single_call(dev, models, front, hop, binarize):
    lf = _lf(models, front, hop, binarize)
    wavs = [w.to(dev) for w in _recordings(LENGTHS, seed=100)]
    durations = [w.numel() / 16000.0 for w in wavs]
    durations[2] += 0.25                                  # a duration that is not the sample count's
    got = lf(wavs, durations=durations)
    assert len(got) == len(wavs)
    for w, d, g in zip(wavs, durations, got):
        _same(g, lf(w, d))
    if hop is None:
        assert got[0]["prob"].shape[0] == 0 and got[0]["stream_dec"].numel() == 0 and got[0]["intervals"] == []
    assert any(len(g["intervals"]) for g in got)


@pytest.mark.parametrize("front,hop,binarize", [("fbank", "overlap", False), ("fbank", None, True), ("sincnet", "overlap", True),
                                                ("sincnet", None, False)])
def test_launch_boundaries(dev, models, front, hop, binarize):
    """max_rows = 7 puts recordings across launches; the results equal one launch of every window."""
    wavs = [w.to(dev) for w in _recordings([302400, 80000, 500000, 272000, 32000, 160000], seed=200)]
    small = _lf(models, front, hop, binarize, max_rows=7)(wavs)
    big = _lf(models, front, hop, binarize, max_rows=4096)(wavs)
    assert sum(g["prob"].shape[0] for g in big) > 7 * 2
    for a, b in zip(small, big):
        _same(a, b)


@pytest.mark.parametrize("front,hop", [("fbank", None), ("fbank", "overlap"), ("sincnet", None), ("sincnet", "overlap")])
def test_int16_input(dev, models, front, hop):
    g = torch.Generator().manual_seed(3)
    pcm = [torch.randint(-12000, 12000, (n,), generator=g, dtype=torch.int16) for n in (302400, 80000, 20000, 991)]
    lf = _lf(models, front, hop, binarize=False)
    got = lf([x.to(dev) for x in pcm])
    want = lf([(x.float() / 32768.0).to(dev) for x in pcm])
    for a, b in zip(got, want):
        _same(a, b)


@pytest.mark.parametrize("front,hop", [("fbank", None), ("fbank", "overlap"), ("sincnet", None), ("sincnet", "overlap")])
def test_rows_never_read_past_their_recording(dev, models, front, hop):
    """Recordings as views of one buffer with NaN samples between them: a row that read one sample beyond its recording (or
    before it) would turn its probabilities into NaN.  Every recording starts 16-byte aligned, as a fresh allocation does."""
    recs = _recordings([302400, 20000, 991, 272000, 80000, 123457], seed=300)
    guard = 64
    starts, pos = [], guard
    for r in recs:
        starts.append(pos)
        pos += r.numel() + guard
        pos += -pos % 4
    buf = torch.full((pos + guard,), float("nan"), device=dev)
    for s, r in zip(starts, recs):
        buf[s:s + r.numel()] = r.to(dev)
    views = [buf[s:s + r.numel()] for s, r in zip(starts, recs)]
    lf = _lf(models, front, hop, binarize=True)
    got = lf(views)
    want = lf([r.to(dev) for r in recs])
    for a, b in zip(got, want):
        assert torch.isfinite(a["prob"]).all()
        _same(a, b)


def test_stitch_center_streams_against_oracle(dev):
    from oracle import longform as olf
    g = np.random.default_rng(11)
    for Tw, hop in ((500, 500), (500, 250), (500, 100), (7, 3), (1, 1)):
        # windows per recording, including none and one, and R = 1
        for W_list in ([3], [0, 1, 5, 2, 0, 9, 1], [int(x) for x in g.integers(0, 6, 40)]):
            lens = []
            for W in W_list:
                full = (W - 1) * hop + Tw if W else 0
                lens.append(int(g.integers(0, full + 3)) if W else int(g.integers(0, 3)))
            prob = g.random((sum(W_list), Tw)).astype(np.float32)
            win_off = np.concatenate([[0], np.cumsum(W_list)]).tolist()
            frame_off = np.concatenate([[0], np.cumsum(lens)]).tolist()
            for src in (prob, (prob > 0.5).astype(np.uint8)):
                got = torch.ops.b200vad.stitch_center_streams(torch.from_numpy(src).to(dev), win_off, frame_off, hop).cpu().numpy()
                assert got.dtype == src.dtype and got.shape == (frame_off[-1],)
                for r, W in enumerate(W_list):
                    seg = got[frame_off[r]:frame_off[r + 1]]
                    if W == 0:
                        assert (seg == 0).all()
                        continue
                    want = olf.stitch_center(src[win_off[r]:win_off[r + 1]], hop, lens[r])
                    assert np.array_equal(seg, want), (Tw, hop, r)
                    if W_list == [3]:
                        one = torch.ops.b200vad.stitch_center(torch.from_numpy(prob).to(dev), hop, lens[0]).cpu().numpy()
                        if src is prob:
                            assert np.array_equal(seg, one)


def test_threshold_median_streams_against_oracle(dev):
    import oracle
    g = np.random.default_rng(12)
    for lens in ([1], [5000], [0, 1, 2, 48, 49, 50, 0, 2047, 2048, 2049, 4097, 3, 25, 24], [int(x) for x in g.integers(0, 300, 60)]):
        x = (g.random(sum(lens)) < 0.5).astype(np.float32) * 0.4 + g.random(sum(lens)).astype(np.float32) * 0.2 + 0.2
        off = np.concatenate([[0], np.cumsum(lens)]).tolist()
        got = torch.ops.b200vad.threshold_median_streams(torch.from_numpy(x).to(dev), off, 0.5, 49).cpu()
        assert got.dtype == torch.uint8 and got.numel() == sum(lens)
        for r, n in enumerate(lens):
            if n == 0:
                continue
            s = torch.from_numpy(x[off[r]:off[r + 1]]).unsqueeze(0)
            want = oracle.median_filter(s, window=0.01)[0]
            assert torch.equal(got[off[r]:off[r + 1]].long(), want), (r, n)
            one = torch.ops.b200vad.threshold_median(s.to(dev), 0.5, 49, False)[0].cpu()
            assert torch.equal(got[off[r]:off[r + 1]], one)


def test_full_size_one_hour_and_200_short(dev, models):
    """One 1 h recording and 200 of 1 s .. 3 min in one call: each equals its own call."""
    g = np.random.default_rng(13)
    lengths = [3600 * 16000] + [int(x) for x in g.integers(16000, 180 * 16000, 200)]
    gen = torch.Generator(device=dev).manual_seed(1)
    wavs = [0.05 * torch.randn(n, device=dev, generator=gen) for n in lengths]
    wavs[0][: lengths[0] // 2] *= torch.sin(torch.arange(lengths[0] // 2, device=dev) * (2 * np.pi * 0.3 / 16000)).abs()
    for hop in (None, "overlap"):
        lf = _lf(models, "fbank", hop, binarize=hop is None)
        got = lf(wavs)
        for w, g1 in zip(wavs, got):
            _same(g1, lf(w))
        assert got[0]["prob"].shape[0] == (720 if hop is None else 1439) and got[0]["stream_dec"].numel() == 360000
