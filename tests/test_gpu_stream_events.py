"""GPU tests of the streaming speech events: b200vad_regions_step at many chunkings, with and without flushes, against the online
reference of stream_events_oracle; its capacity bound; and StreamingVad with events (both front ends, graph and no graph),
end_streams and set_events, compared exactly with the reference and with sessions that track no events."""
import numpy as np
import pytest
import torch

import binarize_oracle as bo
import stream_events_oracle as so
import util

pytestmark = pytest.mark.gpu

LENGTHS = [1, 2, 31, 32, 33, 257, 2049, 4097]


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import b200vad
    b200vad._lib.init(0)
    return torch.device("cuda:0")


# the parameter set and adversarial rows of test_gpu_binarize.py
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


def _chunkings(T, seed):
    g = np.random.default_rng(seed)
    fixed = [[k] * ((T + k - 1) // k) for k in ((2, 31, 32, 33, 2049) if T <= 257 else (31, 32, 33, 2049))]
    mixed, n = [], 0
    while n < T:
        k = int(g.choice([1, 2, 31, 32, 33, int(g.integers(1, 300)), int(g.integers(1, 2050))]))
        mixed.append(k)
        n += k
    out = fixed + [mixed]
    if T <= 257:
        out.append([1] * T)
    return out


def _events(ev, counts):
    ev, counts = ev.cpu(), counts.cpu()
    return [[(int(k), int(f)) for f, k in ev[r, :int(counts[r])].tolist()] for r in range(ev.shape[0])]


def _drive(dev, rows, p, chunks, flush_at=()):
    """regions_step over the chunks; flush every stream after the chunks whose index is in flush_at, and after the last one.
    Returns the per-call events and the reference's."""
    S, T = rows.shape
    x = torch.from_numpy(rows).to(dev)
    state = torch.zeros((S, 5), dtype=torch.int64, device=dev)
    refs = [so.OnlineRegions(*p) for _ in range(S)]
    got, want = [], []
    n = 0
    for i, k in enumerate(chunks):
        k = min(k, T - n)
        fl = i in flush_at or i == len(chunks) - 1
        flush = torch.ones(S, dtype=torch.bool, device=dev) if fl else None
        ev, counts = torch.ops.b200vad.regions_step(x[:, n:n + k].contiguous(), state, *p, flush)
        got.append(_events(ev, counts))
        w = []
        for r in range(S):
            e = refs[r].push(rows[r, n:n + k]) + (refs[r].end() if fl else [])
            w.append([(kind, f) for kind, f, _ in e])
        want.append(w)
        n += k
    assert torch.equal(state.cpu(), torch.zeros((S, 5), dtype=torch.int64))
    return got, want


@pytest.mark.parametrize("T", LENGTHS)
def test_regions_step_matches_online_reference(dev, T):
    for j, p in enumerate(_params(T)):
        rows = _rows(T, p[0], p[1], seed=T * 31 + j)
        for c, chunks in enumerate(_chunkings(T, seed=T + 7 * j)):
            got, want = _drive(dev, rows, p, chunks)
            assert got == want, (T, p, c)
            flush_at = set(range(0, len(chunks), 3))
            got, want = _drive(dev, rows, p, chunks, flush_at)
            assert got == want, (T, p, c, "flush")


def test_regions_step_state_layout_and_partial_flush(dev):
    """stream r of 6 is flushed after the chunks where r is in the mask; the state rows carry (a, last end, group start,
    status, timeline length)"""
    T = 300
    p = (0.6, 0.4, 2, 3, 4, 5)
    rows = _rows(T, p[0], p[1], seed=3)[:6]
    x = torch.from_numpy(rows).to(dev)
    state = torch.zeros((6, 5), dtype=torch.int64, device=dev)
    refs = [so.OnlineRegions(*p) for _ in range(6)]
    g = np.random.default_rng(9)
    n = 0
    while n < T:
        k = int(min(T - n, g.integers(1, 70)))
        mask = g.integers(0, 2, 6).astype(bool)
        ev, counts = torch.ops.b200vad.regions_step(x[:, n:n + k].contiguous(), state, *p, torch.from_numpy(mask).to(dev))
        got = _events(ev, counts)
        for r in range(6):
            e = refs[r].push(rows[r, n:n + k]) + (refs[r].end() if mask[r] else [])
            assert got[r] == [(kind, f) for kind, f, _ in e]
        st = state.cpu()
        for r in range(6):
            ref = refs[r]
            assert int(st[r, 4]) == ref.t and int(st[r, 0]) == ref.h
            status = 0 if ref.gs < 0 else (2 if ref.emitted else 1)
            assert int(st[r, 3]) == status
            if status:
                assert int(st[r, 2]) == ref.gs
                if not ref.h:
                    assert int(st[r, 1]) == ref.last_end
        n += k


@pytest.mark.parametrize("nf", [1, 2, 31, 32, 33, 257, 2049])
def test_capacity_bound_is_exact_and_nothing_is_written_past_it(dev, nf):
    """1 0 1 0 ... with min_on = 0 and gap_break = 1 emits on every frame; an odd nf ends on a start, so the flush adds one:
    nf + 1 events.  Guard words after the buffer stay untouched, and a smaller cap writes only its first entries."""
    import b200vad
    S = 3
    x = torch.from_numpy(np.tile((np.arange(nf) % 2 == 0).astype(np.float32), (S, 1))).to(dev)
    params = b200vad._lib.BinarizeParams(0.5, 0.5, 0, 0, 0, 0)
    full = nf + (nf % 2)
    want = []
    for i in range(nf):
        want.append((i, 1) if i % 2 == 0 else (i, 0))
    if nf % 2:
        want.append((nf, 0))
    for cap in (nf + 1, max(nf // 2, 1)):
        state = torch.zeros((S, 5), dtype=torch.int64, device=dev)
        buf = torch.full((S * cap * 2 + 64,), -7, dtype=torch.int64, device=dev)
        counts = torch.full((S + 4,), -7, dtype=torch.int32, device=dev)
        flush = torch.ones(S, dtype=torch.uint8, device=dev)
        rc = b200vad.lib().b200vad_regions_step(x.data_ptr(), S, nf, nf, params, state.data_ptr(), flush.data_ptr(), buf.data_ptr(),
                                                counts.data_ptr(), cap, torch.cuda.current_stream(dev).cuda_stream)
        assert rc == 0
        torch.cuda.synchronize()
        assert counts[:S].cpu().tolist() == [full] * S and counts[S:].cpu().tolist() == [-7] * 4
        ev = buf[:S * cap * 2].view(S, cap, 2).cpu()
        for r in range(S):
            k = min(cap, full)
            assert [tuple(v) for v in ev[r, :k].tolist()] == want[:k]
            assert bool((ev[r, k:] == -7).all())
        assert bool((buf[S * cap * 2:].cpu() == -7).all())


# ---------------------------------------------------------------- streaming sessions
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


POLICY = dict(onset=0.6, offset=0.4, min_duration_on=0.05, min_duration_off=0.1, pad_onset=0.02, pad_offset=0.03)


def _session(models, front, S, window, graph, **kw):
    import b200vad
    blob, sblob = models[front]
    hop = 270 if sblob is not None else 160
    return b200vad.StreamingVad(blob, 4, num_streams=S, window=window, hop=hop, use_graph=graph, sincnet_packed=sblob, **kw), hop


def _split(ev):
    """(E, 3) [stream, is_start, frame] -> {stream: [(kind, frame)]}"""
    out = {}
    for s, k, f in ev.tolist():
        out.setdefault(s, []).append((k, f))
    return out


@pytest.mark.parametrize("front", ["fbank", "sincnet"])
@pytest.mark.parametrize("graph", [True, False])
def test_streaming_events(dev, models, front, graph):
    import b200vad
    S, window = 4, 16000
    pol = b200vad.Binarize(**POLICY)
    f = pol.frames(b200vad.binarize.mode_step(front == "sincnet")[0])
    p = (f["onset"], f["offset"], f["pad_onset"], f["pad_offset"], f["min_off"], f["min_on"])
    sv, hop = _session(models, front, S, window, graph, events=pol)
    plain, _ = _session(models, front, S, window, graph)
    pushes = window // hop + 40
    audio = util.synth_wave(S, pushes * hop, seed=23)
    refs = [so.OnlineRegions(*p) for _ in range(S)]
    timeline = [[] for _ in range(S)]
    for i in range(pushes):
        chunk = audio[:, i * hop:(i + 1) * hop].contiguous()
        prob, dec, _ = sv.push(chunk)
        prob0, dec0, _ = plain.push(chunk)
        assert torch.equal(prob, prob0) and torch.equal(dec, dec0)
        ev, sec = sv.pop_events()
        want = []
        for r in range(S):
            timeline[r].append(prob[r].numpy())
            want += [(r, k, fr) for k, fr, _ in refs[r].push(prob[r].numpy())]
        assert [tuple(v) for v in ev.tolist()] == want, i
        assert torch.equal(sec, torch.from_numpy(b200vad.binarize.stream_event_seconds(ev[:, 2].numpy(), front == "sincnet", window)))
    sv.end_streams(range(S))
    ev, _ = sv.pop_events()
    assert [tuple(v) for v in ev.tolist()] == [(r, k, fr) for r in range(S) for k, fr, _ in refs[r].end()]
    sv.close(); plain.close()


@pytest.mark.parametrize("graph", [True, False])
def test_streaming_pairs_equal_offline_binarization(dev, models, graph):
    import b200vad
    S, window = 4, 16000
    pol = b200vad.Binarize(**POLICY)
    f = pol.frames(0.01)
    p = (f["onset"], f["offset"], f["pad_onset"], f["pad_offset"], f["min_off"], f["min_on"])
    sv, hop = _session(models, "fbank", S, window, graph, events=pol)
    audio = util.synth_wave(S, 160 * hop, seed=29)
    probs, evs = [], []
    for i in range(160):
        probs.append(sv.push(audio[:, i * hop:(i + 1) * hop].contiguous())[0])
        evs.append(sv.pop_events()[0])
    sv.end_streams([2, 0, 3, 1])
    evs.append(sv.pop_events()[0])
    split = _split(torch.cat(evs))
    x = torch.cat(probs, 1).numpy()
    n_regions = 0
    for r in range(S):
        want = bo.binarize(x[r], *p)[1]
        assert so.pairs(split.get(r, [])) == want, r
        n_regions += len(want)
    assert n_regions > 0
    sv.close()


@pytest.mark.parametrize("front", ["fbank", "sincnet"])
@pytest.mark.parametrize("graph", [True, False])
def test_end_streams_gives_a_fresh_stream(dev, models, front, graph):
    import b200vad
    S, window = 3, 16000
    pol = b200vad.Binarize(**POLICY)
    f = pol.frames(b200vad.binarize.mode_step(front == "sincnet")[0])
    p = (f["onset"], f["offset"], f["pad_onset"], f["pad_offset"], f["min_off"], f["min_on"])
    a, hop = _session(models, front, S, window, graph, events=pol)
    same, _ = _session(models, front, S, window, graph)
    before, after = 30, 25
    audio = util.synth_wave(S, (before + after) * hop, seed=31)
    for i in range(before):
        c = audio[:, i * hop:(i + 1) * hop].contiguous()
        a.push(c); same.push(c)
    a.pop_events()
    a.end_streams([1])
    a.pop_events()
    fresh, _ = _session(models, front, S, window, graph)
    ref = so.OnlineRegions(*p)
    for i in range(before, before + after):
        c = audio[:, i * hop:(i + 1) * hop].contiguous()
        pa, da, _ = a.push(c)
        pf, df, _ = fresh.push(c)
        ps, ds, _ = same.push(c)
        assert torch.equal(pa[1], pf[1]) and torch.equal(da[1], df[1]), i
        for r in (0, 2):
            assert torch.equal(pa[r], ps[r]) and torch.equal(da[r], ds[r]), i
        ev, _ = a.pop_events()
        got1 = [(k, fr) for s, k, fr in ev.tolist() if s == 1]
        assert got1 == [(k, fr) for k, fr, _ in ref.push(pa[1].numpy())]
    w, _, _ = a.snapshot()
    n_new = after * hop
    assert bool((w[1, :window - n_new] == 0).all())
    assert torch.equal(w[1, window - n_new:], audio[1, before * hop:])
    for s in (a, same, fresh):
        s.close()


def test_end_streams_refuses_bad_indices(dev, models):
    import b200vad
    sv, _ = _session(models, "fbank", 3, 16000, False)
    for idx in ([3], [-1], [0, 0], [1, 2, 1]):
        with pytest.raises(b200vad._lib.B200VadError):
            sv.end_streams(idx)
    sv.end_streams([])
    sv.close()


@pytest.mark.parametrize("graph", [True, False])
def test_set_events_switches_policy_mid_stream(dev, models, graph):
    import b200vad
    S, window = 3, 16000
    pols = [b200vad.Binarize(**POLICY), b200vad.Binarize(onset=0.7, offset=0.2, min_duration_on=0.0, min_duration_off=0.3,
                                                         pad_onset=0.05, pad_offset=0.0)]
    ps = []
    for pol in pols:
        f = pol.frames(0.01)
        ps.append((f["onset"], f["offset"], f["pad_onset"], f["pad_offset"], f["min_off"], f["min_on"]))
    sv, hop = _session(models, "fbank", S, window, graph, events=pols[0])
    n1, n2, n3 = 120, 90, 20
    audio = util.synth_wave(S, (n1 + n2 + n3) * hop, seed=37)
    push = lambda i: sv.push(audio[:, i * hop:(i + 1) * hop].contiguous())[0]
    probs, evs = [], []
    for i in range(n1):
        probs.append(push(i))
    sv.set_events(pols[1])
    for i in range(n1, n1 + n2):
        probs.append(push(i))
    sv.set_events(None)
    evs = sv.pop_events()[0]
    for i in range(n1 + n2, n1 + n2 + n3):
        push(i)
    assert sv.pop_events()[0].shape == (0, 3)
    split = _split(evs)
    x = torch.cat(probs, 1).numpy()
    for r in range(S):
        want = bo.binarize(x[r, :n1], *ps[0])[1] + [(s + n1, e + n1) for s, e in bo.binarize(x[r, n1:], *ps[1])[1]]
        assert so.pairs(split.get(r, [])) == want, r
    sv.close()


def test_config5_shape_with_events(dev, models):
    import b200vad
    blob, _ = models["fbank"]
    sv = b200vad.StreamingVad(blob, 4, num_streams=256, window=80000, hop=160, events=b200vad.Binarize(**POLICY))
    gen = torch.Generator().manual_seed(0)
    chunks = [(0.1 * torch.randn(256, 160, generator=gen)).pin_memory() for _ in range(8)]
    ms = []
    n = 0
    for i in range(60):
        prob, dec, t = sv.push(chunks[i % 8])
        assert prob.shape == (256, 1) and dec.shape == (256, 1)
        ms.append(t)
        ev, sec = sv.pop_events()
        assert ev.shape[1] == 3 and sec.shape == (ev.shape[0],) and ev.shape[0] <= 256
        n += ev.shape[0]
    ms = sorted(ms[10:])
    print(f"config 5 with events: push p50 {ms[len(ms) // 2]:.3f} ms, max {ms[-1]:.3f} ms, {n} events in 60 pushes")
    sv.close()
