"""GPU tests of the binarization (onset / offset hysteresis, pads, minimum durations): the b200vad_binarize kernels over their
whole parameter range at every word and chunk edge, its output cap, and every mode that takes it (whole-path op, host session,
streaming, long form), all compared with torch.equal against the frame-domain reference in binarize_oracle."""
import math

import numpy as np
import pytest
import torch

import binarize_oracle as bo
import util

pytestmark = pytest.mark.gpu

EINVAL = -1
# word (32) and chunk (2048 frames = 64 words) edges of the kernel and a model row (800); the 1 h stream has a test of its own
LENGTHS = [1, 2, 31, 32, 33, 255, 256, 257, 800, 2047, 2048, 2049, 4097]


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import b200vad
    b200vad._lib.init(0)
    return torch.device("cuda:0")


def _params(T):
    big = T + 5
    return [(0.5, 0.5, 0, 0, 0, 0), (0.6, 0.4, 0, 0, 0, 0), (0.6, 0.4, 1, 1, 1, 1), (0.6, 0.4, 2, 0, 2, 0), (0.6, 0.4, 0, 2, 0, 2),
            (0.55, 0.45, big, big, big, big), (0.7, 0.3, 0, 0, big, 0), (0.7, 0.3, 0, 0, 0, big), (0.7, 0.3, 3, 5, 7, 11),
            (0.5, 0.2, 1, 0, 40, 3)]


def _rows(T, onset, offset, seed):
    """(8, T) float32: a random walk around the thresholds, runs of onset / offset and their adjacent floats, NaN / +-inf runs,
    all zero, all one, alternating 1 0 1 0 ..., uniform noise"""
    g = np.random.default_rng(seed)
    on, off = np.float32(onset), np.float32(offset)
    near = np.array([on, np.nextafter(on, np.float32(2)), np.nextafter(on, np.float32(-2)), off, np.nextafter(off, np.float32(2)),
                     np.nextafter(off, np.float32(-2))], np.float32)
    special = np.array([np.nan, np.inf, -np.inf, 0.5, on, off], np.float32)
    runs = lambda vals: np.repeat(g.choice(vals, T), g.integers(1, 9, T))[:T]
    rows = np.empty((8, T), np.float32)
    rows[0] = 0.5 + 0.1 * np.cumsum(g.standard_normal(T))
    rows[1] = runs(near)
    rows[2] = runs(special)
    rows[3] = 0.0
    rows[4] = 1.0
    rows[5] = (np.arange(T) % 2 == 0)
    rows[6] = g.uniform(0, 1, T)
    rows[7] = runs(np.concatenate([near, special]))
    return rows


def _ref(rows, p, row_ids=None):
    decs, segs = [], []
    for i, x in enumerate(rows):
        d, regions = bo.binarize(x, *p)
        decs.append(torch.from_numpy(d))
        segs += [(i if row_ids is None else row_ids[i], s, e - 1) for s, e in regions]
    return decs, torch.tensor(segs, dtype=torch.int32).reshape(-1, 3)


@pytest.mark.parametrize("T", LENGTHS)
def test_op_uniform_rows(dev, T):
    for j, p in enumerate(_params(T)):
        rows = _rows(T, p[0], p[1], seed=T * 31 + j)
        dec, seg, counts = torch.ops.b200vad.binarize(torch.from_numpy(rows).to(dev), None, *p)
        want_dec, want_seg = _ref(rows, p)
        assert torch.equal(dec.cpu(), torch.stack(want_dec)), (T, p)
        assert torch.equal(seg.cpu(), want_seg), (T, p)
        assert torch.equal(counts.cpu(), torch.bincount(want_seg[:, 0].long(), minlength=8).int()), (T, p)


@pytest.mark.parametrize("seed", [0, 1])
def test_op_ragged_with_empty_streams(dev, seed):
    g = np.random.default_rng(seed)
    lens = [0, 1, 2049, 0, 33, 4096, 0, 31, 800, 257, 0]
    for j, p in enumerate(_params(max(lens))):
        streams = [_rows(n, p[0], p[1], seed=seed * 100 + j + n)[g.integers(8)] if n else np.empty(0, np.float32) for n in lens]
        flat = np.concatenate(streams).astype(np.float32)
        offs = torch.tensor(np.concatenate([[0], np.cumsum(lens)]), dtype=torch.int64)
        dec, seg, counts = torch.ops.b200vad.binarize(torch.from_numpy(flat).to(dev), offs.to(dev), *p)
        want_dec, want_seg = _ref(streams, p)
        assert torch.equal(dec.cpu(), torch.cat(want_dec)), p
        assert torch.equal(seg.cpu(), want_seg), p
        assert torch.equal(counts.cpu(), torch.bincount(want_seg[:, 0].long(), minlength=len(lens)).int()), p


@pytest.mark.parametrize("p", [(0.6, 0.4, 0, 0, 0, 0), (0.6, 0.4, 25, 40, 100, 50), (0.5, 0.5, 360005, 0, 0, 0),
                               (0.7, 0.2, 0, 0, 360005, 0)])
def test_op_one_hour_stream(dev, p):
    T = 360000
    g = np.random.default_rng(7)
    x = ((0.05 * np.cumsum(g.standard_normal(T))) % 1.0).astype(np.float32)     # a random walk folded into [0, 1)
    x[1000:1500] = np.nan
    dec, seg, _ = torch.ops.b200vad.binarize(torch.from_numpy(x).to(dev).view(1, -1), None, *p)
    want_dec, want_seg = _ref([x], p)
    assert torch.equal(dec.cpu()[0], want_dec[0]) and torch.equal(seg.cpu(), want_seg)


@pytest.mark.parametrize("T", LENGTHS)
def test_alternating_fills_cap_exactly_and_writes_nothing_past_it(dev, T):
    import b200vad
    R = 3
    x = torch.from_numpy(np.tile((np.arange(T) % 2 == 0).astype(np.float32), (R, 1))).to(dev)
    per = (T + 1) // 2
    params = b200vad._lib.BinarizeParams(0.5, 0.5, 0, 0, 0, 0)
    for cap in (R * per, R * per - 1, per // 2):
        dec = torch.full((R, T), 7, dtype=torch.uint8, device=dev)
        counts = torch.empty(R, dtype=torch.int32, device=dev)
        seg_off = torch.empty(R + 1, dtype=torch.int64, device=dev)
        seg = torch.full((R * per + 8, 3), -5, dtype=torch.int32, device=dev)
        rc = b200vad.lib().b200vad_binarize(x.data_ptr(), None, R, T, params, dec.data_ptr(), counts.data_ptr(), seg_off.data_ptr(),
                                            seg.data_ptr(), cap, torch.cuda.current_stream(dev).cuda_stream)
        assert rc == 0
        torch.cuda.synchronize()
        assert counts.cpu().tolist() == [per] * R and seg_off.cpu().tolist() == [i * per for i in range(R + 1)]
        want = torch.tensor([(r, 2 * i, 2 * i) for r in range(R) for i in range(per)], dtype=torch.int32)
        assert torch.equal(seg[:cap].cpu(), want[:cap])
        assert bool((seg[max(cap, 0):].cpu() == -5).all())                   # nothing past cap
        if cap >= R * per:
            assert torch.equal(dec.cpu(), (x.cpu() > 0.5).to(torch.uint8))


def test_invalid_params_refused(dev):
    import b200vad
    P = b200vad._lib.BinarizeParams
    x = torch.zeros((1, 4), device=dev)
    dec = torch.empty((1, 4), dtype=torch.uint8, device=dev)
    counts = torch.empty(1, dtype=torch.int32, device=dev)
    seg_off = torch.empty(2, dtype=torch.int64, device=dev)
    seg = torch.empty((2, 3), dtype=torch.int32, device=dev)
    for p in (P(0.4, 0.5, 0, 0, 0, 0), P(float("nan"), 0.5, 0, 0, 0, 0), P(0.5, float("-inf"), 0, 0, 0, 0), P(0.5, 0.5, -1, 0, 0, 0),
              P(0.5, 0.5, 0, -1, 0, 0), P(0.5, 0.5, 0, 0, -1, 0), P(0.5, 0.5, 0, 0, 0, -1)):
        rc = b200vad.lib().b200vad_binarize(x.data_ptr(), None, 1, 4, p, dec.data_ptr(), counts.data_ptr(), seg_off.data_ptr(),
                                            seg.data_ptr(), 2, None)
        assert rc == EINVAL
    assert b200vad.lib().b200vad_binarize(x.data_ptr(), None, 1, 4, None, dec.data_ptr(), counts.data_ptr(), seg_off.data_ptr(),
                                          seg.data_ptr(), 2, None) == EINVAL


# ---------------------------------------------------------------- whole path, sessions, streaming, long form
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


POLICY = (0.6, 0.4, 3, 5, 8, 10)                # frames: onset, offset, pad_onset, pad_offset, min_off, min_on


def _default(wav, blob, sblob):
    if sblob is None:
        return torch.ops.b200vad.vad_pipeline(wav, None, blob, 4, 0.5, 49)
    return torch.ops.b200vad.vad_pipeline_sincnet(wav, blob, sblob, 4, 0.5, 49)


@pytest.mark.parametrize("front", ["fbank", "sincnet"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.int16])
def test_whole_path(dev, models, front, dtype):
    blob, sblob = models[front]
    wav = util.synth_wave(37, 48123, seed=11)
    if dtype == torch.int16:
        wav = (wav * 32767).round().clamp(-32768, 32767).to(torch.int16)
    wav = wav.to(dev)
    prob, dec, seg, counts = torch.ops.b200vad.vad_pipeline_binarize(wav, None, blob, sblob, 4, *POLICY)
    assert torch.equal(prob, _default(wav, blob, sblob)[0])
    d, s, c = torch.ops.b200vad.binarize(prob, None, *POLICY)
    assert torch.equal(dec, d) and torch.equal(seg, s) and torch.equal(counts, c)
    want_dec, want_seg = _ref(prob.cpu().numpy(), POLICY)
    assert torch.equal(dec.cpu(), torch.stack(want_dec)) and torch.equal(seg.cpu(), want_seg)
    pp, pd, pseg, pc, poff = torch.ops.b200vad.vad_pipeline_binarize_padded(wav, None, blob, sblob, 4, *POLICY)
    T = prob.shape[1]
    assert pseg.shape == (37 * ((T + 1) // 2), 3) and int(poff[-1]) == seg.shape[0]
    assert torch.equal(pp, prob) and torch.equal(pd, dec) and torch.equal(pseg[: seg.shape[0]], seg) and torch.equal(pc, counts)


@pytest.mark.parametrize("front", ["fbank", "sincnet"])
def test_host_session(dev, models, front):
    import b200vad
    blob, sblob = models[front]
    N, B = 48123, 9
    wav = util.synth_wave(2 * B, N, seed=13)
    pol = b200vad.Binarize(onset=0.6, offset=0.4, min_duration_on=0.1, min_duration_off=0.08, pad_onset=0.03, pad_offset=0.05)
    step, _ = b200vad.binarize.mode_step(sblob is not None)
    f = pol.frames(step)
    sess = b200vad.HostSession(blob, 4, N, chunk_rows=B, sincnet_packed=sblob, binarize=pol)
    plain = b200vad.HostSession(blob, 4, N, chunk_rows=B, sincnet_packed=sblob)
    outs = [sess.submit(i, wav[i * B:(i + 1) * B].contiguous().pin_memory(), want_prob=True) for i in range(2)]
    for i in range(2):
        got = sess.wait(i, outs[i])
        prob, dec, seg, _ = torch.ops.b200vad.vad_pipeline_binarize(wav[i * B:(i + 1) * B].to(dev), None, blob, sblob, 4,
                                                                     f["onset"], f["offset"], f["pad_onset"], f["pad_offset"],
                                                                     f["min_off"], f["min_on"])
        assert torch.equal(got["prob"], prob.cpu()) and torch.equal(got["dec"], dec.cpu()) and torch.equal(got["seg"], seg.cpu())
    sess.set_binarize(None)
    for s in (sess, plain):
        o = s.submit(0, wav[:B].contiguous().pin_memory(), want_prob=True)
        s.wait(0, o)
        if s is sess:
            first = {k: o[k].clone() for k in ("dec", "prob", "seg")}
    for k in ("dec", "prob", "seg"):
        assert torch.equal(first[k], o[k])
    sess.close(); plain.close()


def _bin_rows(prob, f):
    return torch.ops.b200vad.binarize(prob, None, f["onset"], f["offset"], f["pad_onset"], f["pad_offset"], f["min_off"], f["min_on"])


@pytest.mark.parametrize("front", ["fbank", "sincnet"])
@pytest.mark.parametrize("graph", [True, False])
def test_streaming(dev, models, front, graph):
    import b200vad
    blob, sblob = models[front]
    S, window = 4, 16000
    hop = 270 if sblob is not None else 160
    step, _ = b200vad.binarize.mode_step(sblob is not None)
    pols = [b200vad.Binarize(onset=0.6, offset=0.4, min_duration_on=0.05, pad_offset=0.02),
            b200vad.Binarize(onset=0.7, offset=0.2, min_duration_off=0.2, pad_onset=0.05)]
    sv = b200vad.StreamingVad(blob, 4, num_streams=S, window=window, hop=hop, use_graph=graph, sincnet_packed=sblob, binarize=pols[0])
    total = util.synth_wave(S, window + 20 * hop, seed=17)
    fed = 0
    for i in range(window // hop + 6):
        if i == window // hop:
            sv.set_binarize(pols[1])                        # takes effect on the next push
        pol = pols[0] if i < window // hop else pols[1]
        prob, dec, _ = sv.push(total[:, fed:fed + hop].contiguous(), thr=0.3, kernel=3)   # thr / kernel are ignored
        fed += hop
        if i in (3, window // hop - 1, window // hop, window // hop + 5):
            _, p_all, d_all = sv.snapshot()
            want, _, _ = _bin_rows(p_all.to(dev), pol.frames(step))
            assert torch.equal(d_all, want.cpu()) and torch.equal(dec, want[:, -sv.nf:].cpu())
            assert torch.equal(prob, p_all[:, -sv.nf:])
    sv.set_binarize(None)
    prob, dec, _ = sv.push(total[:, fed:fed + hop].contiguous())
    _, p_all, d_all = sv.snapshot()
    assert torch.equal(d_all, torch.ops.b200vad.threshold_median(p_all.to(dev), 0.5, 49, False).cpu())
    sv.close()


@pytest.mark.parametrize("front", ["fbank", "sincnet"])
@pytest.mark.parametrize("hop", [None, 270 * 120])
def test_longform(dev, models, front, hop):
    import b200vad
    from b200vad.host import fbank_num_frames, get_num_frames
    blob, sblob = models[front]
    sinc = sblob is not None
    if hop is not None and not sinc:
        hop = 160 * 200
    seconds = 18.9                                    # a 3.9 s ragged last window
    N = int(seconds * 16000)
    wav = util.synth_wave(1, N, seed=19)[0].to(dev)
    pol = b200vad.Binarize(onset=0.6, offset=0.4, min_duration_on=0.2, min_duration_off=0.3, pad_onset=0.05, pad_offset=0.1)
    res = b200vad.LongFormVad(blob, 4, hop=hop, sincnet_packed=sblob, binarize=pol)(wav)
    step, t0 = b200vad.binarize.mode_step(sinc)
    f = pol.frames(step)
    prob = res["prob"]
    if hop is None:
        n = math.ceil(get_num_frames(16000 * seconds)) + 1 if sinc else math.ceil(seconds / 0.01) + 1
        stream = prob.reshape(-1)[: min(n, prob.numel())]
    else:
        L = get_num_frames(N) if sinc else fbank_num_frames(N)
        stream = torch.ops.b200vad.stitch_center(prob, hop // (270 if sinc else 160), L)
    dec, regions = bo.binarize(stream.cpu().numpy(), f["onset"], f["offset"], f["pad_onset"], f["pad_offset"], f["min_off"], f["min_on"])
    assert torch.equal(res["stream_dec"].cpu(), torch.from_numpy(dec))
    assert res["intervals"] == [[s * step + t0, min(e * step + t0, seconds)] for s, e in regions]
    assert len(regions) > 0
