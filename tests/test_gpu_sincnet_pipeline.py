"""GPU tests of the SincNet -> PyanNet whole path (the reference's feature_extractor="sincnet" flow): the one-call device
pipeline against the drop-in VadModel('PyanNet') and the oracle, 16-bit PCM input, the padded op, the host session, the
long-form modes and streaming."""

import pytest
import torch

import util

pytestmark = pytest.mark.gpu

K = 49          # median window of PyanNet: vad_engine.py:207 uses window 0.01 when encoding_dim != 768


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import b200vad
    b200vad._lib.init(0)
    return torch.device("cuda:0")


def _pyannet(dev, wav_for_spread, sigma=2.0):
    """oracle PyanNet, the drop-in VadModel('PyanNet') with the same weights, and the two packed blobs"""
    import b200vad
    from src.engines import VadModel
    o = util.make_oracle("PyanNet", {}, spread=True, feats=wav_for_spread, sigma=sigma)
    m = VadModel("PyanNet", {}).eval()
    m.load_state_dict(o.state_dict())
    m = m.to(dev)
    sd = o.model.state_dict()
    blob = b200vad.pack_model({k: v for k, v in sd.items() if not k.startswith("sincnet.")}, dev, 60, 4)
    sblob = b200vad.pack_sincnet(sd, dev)
    return o, m, blob, sblob


def _dropin(m, wav):
    """the current composition: VadModel('PyanNet') forward, then threshold / median and segments with min_run = 1"""
    with torch.no_grad():
        prob = m(wav.unsqueeze(1)).squeeze(-1)
    dec = torch.ops.b200vad.threshold_median(prob, 0.5, K, False)
    seg, counts = torch.ops.b200vad.segments(dec, None, 1)
    return prob, dec, seg, counts


def _assert_same(a, b):
    for x, y in zip(a, b):
        assert x.shape == y.shape and torch.equal(x, y)


@pytest.fixture(scope="module")
def model(dev):
    return _pyannet(dev, util.synth_wave(4, 80000, seed=71))


# ---------------------------------------------------------------- pipeline == drop-in model
@pytest.mark.parametrize("B", [1, 37, 65])
@pytest.mark.parametrize("N", [80000, 128000, 48123])
def test_pipeline_equals_dropin(dev, model, B, N):
    _, m, blob, sblob = model
    wav = util.synth_wave(B, N, seed=B * 7 + N % 97).to(dev)
    got = torch.ops.b200vad.vad_pipeline_sincnet(wav, blob, sblob, 4, 0.5, K)
    want = _dropin(m, wav)
    _assert_same(got, want)
    import b200vad
    assert got[0].shape == (B, b200vad.host.get_num_frames(N))


def test_pipeline_equals_dropin_many_frontend_chunks(dev, model):
    """700 x 8 s is more than one front-end chunk (651 rows at 8 s): every chunk writes its rows into one planes buffer and
    the LSTM layers run over the whole batch."""
    _, m, blob, sblob = model
    wav = util.synth_wave(700, 128000, seed=17).to(dev)
    _assert_same(torch.ops.b200vad.vad_pipeline_sincnet(wav, blob, sblob, 4, 0.5, K), _dropin(m, wav))


def test_pipeline_small_workspace_chunks_the_model(dev, model):
    """A workspace that holds the planes of the whole batch but the LSTM stack for only 64 sequences at a time."""
    import b200vad
    _, m, blob, sblob = model
    B, N = 150, 48123
    wav = util.synth_wave(B, N, seed=23).to(dev)
    lib = b200vad._lib.lib()
    Ts = lib.b200vad_sincnet_num_frames(N)
    ws_bytes = 256 * B * Ts + lib.b200vad_pipeline_sincnet_workspace_bytes(1, N)
    assert ws_bytes < lib.b200vad_pipeline_sincnet_workspace_bytes(B, N) // 2
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    cap = B * ((Ts + 1) // 2)
    prob = torch.empty((B, Ts), dtype=torch.float32, device=dev)
    dec = torch.empty((B, Ts), dtype=torch.uint8, device=dev)
    counts = torch.empty(B, dtype=torch.int32, device=dev)
    seg_off = torch.empty(B + 1, dtype=torch.int64, device=dev)
    seg = torch.empty((cap, 3), dtype=torch.int32, device=dev)
    b200vad._lib.check(lib.b200vad_pipeline_sincnet_f32(blob.data_ptr(), sblob.data_ptr(), 4, wav.data_ptr(), B, N, N, 0.5, K,
                                                        prob.data_ptr(), dec.data_ptr(), counts.data_ptr(), seg_off.data_ptr(),
                                                        seg.data_ptr(), cap, ws.data_ptr(), ws_bytes,
                                                        torch.cuda.current_stream(dev).cuda_stream), "pipeline_sincnet_f32")
    n = int(seg_off[-1].item())
    _assert_same((prob, dec, seg[:n], counts), _dropin(m, wav))


# ---------------------------------------------------------------- against the fp32 oracle
def test_full_size_pipeline_against_oracle(dev):
    """1024 x 8 s: 16 random rows of the one-call pipeline against the CPU oracle PyanNet."""
    import oracle
    B, N = 1024, 128000
    wav = util.synth_wave(B, N, seed=33)
    rows = torch.randperm(B, generator=torch.Generator().manual_seed(4))[:16]
    sub = wav[rows]
    o, _, blob, sblob = _pyannet(dev, sub)
    with torch.no_grad():
        ref_p = o(sub.unsqueeze(1)).squeeze(-1)
    ref_d = oracle.median_filter(ref_p, window=0.01)
    prob, dec, _, _ = torch.ops.b200vad.vad_pipeline_sincnet(wav.to(dev), blob, sblob, 4, 0.5, K)
    p = prob[rows.to(dev)].cpu()
    d = dec[rows.to(dev)].cpu().long()
    err = util.prob_err(p, ref_p)
    near = (ref_p - 0.5).abs() <= util.NEAR_THR
    diff = d != ref_d
    print(f"SincNet pipeline 1024 x 8 s, 16 rows vs oracle: rel err of p {err:.2e}; near-threshold frames {int(near.sum())}; "
          f"decisions differing {int(diff.sum())}")
    assert err <= util.PROB_RTOL, err
    for b, t in zip(*torch.nonzero(diff, as_tuple=True)):
        assert near[b, max(0, int(t) - K // 2): int(t) + K // 2 + 1].any(), (int(b), int(t))


# ---------------------------------------------------------------- int16 PCM, padded form
def _pcm(B, N, seed):
    w = util.synth_wave(B, N, seed=seed)
    return (w * 32767.0).round().clamp(-32768, 32767).to(torch.int16)


@pytest.mark.parametrize("B,N", [(37, 48123), (5, 128000)])
def test_int16_equals_float(dev, model, B, N):
    _, _, blob, sblob = model
    w16 = _pcm(B, N, seed=B + 1).to(dev)
    got = torch.ops.b200vad.vad_pipeline_sincnet(w16, blob, sblob, 4, 0.5, K)
    want = torch.ops.b200vad.vad_pipeline_sincnet(w16.float() / 32768, blob, sblob, 4, 0.5, K)
    _assert_same(got, want)


def test_padded_matches_exact(dev, model):
    _, _, blob, sblob = model
    wav = util.synth_wave(37, 48000, seed=5).to(dev)
    p1, d1, s1, c1 = torch.ops.b200vad.vad_pipeline_sincnet(wav, blob, sblob, 4, 0.5, K)
    p2, d2, s2, c2, off = torch.ops.b200vad.vad_pipeline_sincnet_padded(wav, blob, sblob, 4, 0.5, K)
    n = int(off[-1].item())
    Ts = p1.shape[1]
    assert torch.equal(p1, p2) and torch.equal(d1, d2) and torch.equal(c1, c2)
    assert s2.shape == (37 * ((Ts + 1) // 2), 3)
    assert n == s1.shape[0] and torch.equal(s1, s2[:n]) and n > 0
    assert off.shape == (38,) and torch.equal(off[1:] - off[:-1], c1.long())


def test_padded_with_segment_gatherer(dev, model):
    import b200vad
    _, _, blob, sblob = model
    wav = util.synth_wave(20, 48000, seed=6).to(dev)
    g = b200vad.SegmentGatherer(dev)
    want = []
    for b0 in (0, 10):
        _, _, s, _, off = torch.ops.b200vad.vad_pipeline_sincnet_padded(wav[b0:b0 + 10], blob, sblob, 4, 0.5, K)
        g.push(s, off, b0)
        _, _, e, _ = torch.ops.b200vad.vad_pipeline_sincnet(wav[b0:b0 + 10], blob, sblob, 4, 0.5, K)
        e = e.clone()
        e[:, 0] += b0
        want.append(e)
    got = g.drain()
    assert len(got) == 2 and all(torch.equal(a, b) for a, b in zip(got, want))


# ---------------------------------------------------------------- host session
def _session_equals_device(sess, wav_host, blob, sblob, dev, thr=0.5, kernel=K):
    B = wav_host.shape[0]
    want = torch.ops.b200vad.vad_pipeline_sincnet(wav_host.to(dev), blob, sblob, 4, thr, kernel)
    r = sess.run(wav_host, thr, kernel, want_prob=True) if wav_host.dtype == torch.float32 else None
    if r is not None:
        assert torch.equal(r["prob"][:B], want[0].cpu()) and torch.equal(r["dec"][:B], want[1].cpu())
        assert torch.equal(r["seg"], want[2].cpu())
    return want


@pytest.mark.parametrize("dtype", [torch.float32, torch.int16])
def test_session_equals_device_pipeline(dev, model, dtype):
    import b200vad
    _, _, blob, sblob = model
    N, chunk = 80000, 16
    sess = b200vad.HostSession(blob, 4, N, chunk_rows=chunk, sincnet_packed=sblob)
    assert sess.T == b200vad.host.get_num_frames(N)
    if dtype == torch.float32:
        wav = util.synth_wave(2 * chunk + 5, N, seed=41).pin_memory()      # run(): three chunks through both slots
        _session_equals_device(sess, wav, blob, sblob, dev)
    # submit / wait, two slots in flight, B = 1 and B = chunk_rows
    batches = []
    for i, B in enumerate((1, chunk, chunk, 1)):
        w = util.synth_wave(B, N, seed=50 + i)
        if dtype == torch.int16:
            w = (w * 32767.0).round().clamp(-32768, 32767).to(torch.int16)
        batches.append(w.pin_memory())
    outs = [dict(), dict()]
    for i, w in enumerate(batches):
        slot = i & 1
        if i >= 2:
            _check_slot(sess, slot, outs[slot], batches[i - 2], blob, sblob, dev)
        sess.submit(slot, w, 0.5, K, want_dec=True, want_prob=True, out=outs[slot])
    for i in (len(batches) - 2, len(batches) - 1):
        _check_slot(sess, i & 1, outs[i & 1], batches[i], blob, sblob, dev)
    sess.close()


def _check_slot(sess, slot, out, w, blob, sblob, dev):
    sess.wait(slot, out)
    x = w.to(dev)
    p, d, s, _ = torch.ops.b200vad.vad_pipeline_sincnet(x if x.dtype == torch.float32 else x.float() / 32768, blob, sblob, 4, 0.5, K)
    assert torch.equal(out["prob"], p.cpu()) and torch.equal(out["dec"], d.cpu()) and torch.equal(out["seg"], s.cpu())


def test_session_single_frame_runs(dev, model):
    """A pulse train with a period of two SincNet frames (540 samples) makes neighbouring frames differ; with the threshold
    between the even- and odd-frame levels and no median filter (kernel 1) rows hold single-frame runs, which the SincNet RLE
    keeps (min_run 1) and the session must return as the device pipeline does."""
    import b200vad
    _, _, blob, sblob = model
    N, B = 48000, 8
    t = torch.arange(N)
    g = torch.Generator().manual_seed(3)
    wav = ((t % 540) < 120).float() * (0.5 + 0.05 * torch.randn(B, N, generator=g)) + 0.01 * torch.randn(B, N, generator=g)
    p, _, _, _ = torch.ops.b200vad.vad_pipeline_sincnet(wav.to(dev), blob, sblob, 4, 0.5, 1)
    mid = p[:, p.shape[1] // 4: 3 * p.shape[1] // 4].cpu()
    thr = float(0.5 * (mid[:, 0::2].median() + mid[:, 1::2].median()))
    Ts = p.shape[1]
    sess = b200vad.HostSession(blob, 4, N, chunk_rows=B, sincnet_packed=sblob)
    want = _session_equals_device(sess, wav.pin_memory(), blob, sblob, dev, thr=thr, kernel=1)
    seg, counts = want[2].cpu(), want[3].cpu()
    print(f"single-frame runs: {int((seg[:, 1] == seg[:, 2]).sum())} of {seg.shape[0]} segments; max per row {int(counts.max())} "
          f"(capacity ceil(T/2) = {(Ts + 1) // 2})")
    assert bool((seg[:, 1] == seg[:, 2]).any())
    sess.close()


# ---------------------------------------------------------------- long-form
@pytest.mark.parametrize("seconds", [21.0, 18.9, 17.0])      # full windows only / 3.9 s tail kept / 2 s tail dropped
def test_longform_reference_semantics(dev, seconds):
    import b200vad
    import oracle
    from oracle import longform as olf
    N = int(seconds * 16000)
    wav = util.synth_wave(1, N, seed=int(seconds * 10))[0]
    o, _, blob, sblob = _pyannet(dev, wav[:80000].unsqueeze(0))
    res = b200vad.LongFormVad(blob, 4, sincnet_packed=sblob)(wav.to(dev))
    wins = olf.cut_windows(N)
    assert res["windows"] == wins
    rows = torch.zeros(len(wins), 80000)                     # the tail window is zero padded in audio
    for i, (s, n) in enumerate(wins):
        rows[i, :n] = wav[s:s + n]
    with torch.no_grad():
        ref_prob = o(rows.unsqueeze(1)).squeeze(-1)
    assert util.prob_err(res["prob"].cpu(), ref_prob) <= util.PROB_RTOL
    dur = N / 16000.0
    dec = oracle.median_filter(res["prob"].cpu(), window=0.01)
    stream = oracle.slice_recordings(dec.reshape(-1), [dur], sincnet=True)[0]
    assert torch.equal(res["stream_dec"].cpu().long(), stream)
    want = oracle.merge_intervals_with_buffer(oracle.rle_segments_sincnet(stream.tolist(), dur), dur, 0)
    assert [list(x) for x in res["intervals"]] == [list(x) for x in want]


@pytest.mark.parametrize("hop", [40500, 16200])
def test_longform_overlap_stitching(dev, hop):
    import b200vad
    import oracle
    from oracle import longform as olf
    N = 16000 * 23 + 1234
    wav = util.synth_wave(1, N, seed=hop)[0]
    o, _, blob, sblob = _pyannet(dev, wav[:80000].unsqueeze(0))
    res = b200vad.LongFormVad(blob, 4, hop=hop, sincnet_packed=sblob)(wav.to(dev))
    wins = olf.cut_windows(N, 80000, hop)
    assert res["windows"] == wins
    for i in (0, len(wins) - 1):
        s, n = wins[i]
        row = torch.zeros(1, 80000)
        row[0, :n] = wav[s:s + n]
        with torch.no_grad():
            ref = o(row.unsqueeze(1)).squeeze()
        assert util.prob_err(res["prob"][i].cpu(), ref) <= util.PROB_RTOL
    L = b200vad.host.get_num_frames(N)
    stitched = olf.stitch_center(res["prob"].cpu().numpy(), hop // 270, L)
    dec = oracle.median_filter(torch.from_numpy(stitched).unsqueeze(0), window=0.01)[0]
    assert torch.equal(res["stream_dec"].cpu().long(), dec)
    dur = N / 16000.0
    want = oracle.merge_intervals_with_buffer(oracle.rle_segments_sincnet(dec.tolist(), dur), dur, 0)
    assert [list(x) for x in res["intervals"]] == [list(x) for x in want]
    with pytest.raises(ValueError):
        b200vad.LongFormVad(blob, 4, hop=hop + 160, sincnet_packed=sblob)


# ---------------------------------------------------------------- streaming
@pytest.mark.parametrize("S,window,hop,graph", [(5, 16000, 270, True), (5, 16000, 270, False), (3, 8000, 540, True),
                                                (3, 8000, 540, False)])
def test_streaming_matches_batch_on_buffered_window(dev, model, S, window, hop, graph):
    import b200vad
    _, _, blob, sblob = model
    total = util.synth_wave(S, window + 40 * hop, seed=window + hop)
    sv = b200vad.StreamingVad(blob, 4, num_streams=S, window=window, hop=hop, use_graph=graph, sincnet_packed=sblob)
    nf = hop // 270
    assert sv.nf == nf and sv.T == b200vad.host.get_num_frames(window)
    fed = 0
    steps = window // hop + 7
    for step in range(steps):
        chunk = total[:, fed:fed + hop].contiguous()
        prob, dec, _ = sv.push(chunk if step % 2 else chunk.to(dev))
        fed += hop
        if step in (0, 3, window // hop - 1, steps - 1):
            buf = torch.zeros(S, window)
            n = min(fed, window)
            buf[:, window - n:] = total[:, fed - n:fed]
            w, p_all, d_all = sv.snapshot()
            assert torch.equal(w, buf)                                             # ring buffer == last `window` samples
            bp, bd, _, _ = torch.ops.b200vad.vad_pipeline_sincnet(buf.to(dev), blob, sblob, 4, 0.5, K)
            assert torch.equal(p_all, bp.cpu()) and torch.equal(d_all, bd.cpu())
            assert prob.shape == (S, nf)
            assert torch.equal(prob, bp[:, -nf:].cpu()) and torch.equal(dec, bd[:, -nf:].cpu())
    sv.close()
