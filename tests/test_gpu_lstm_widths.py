"""The LSTM stack at every kind of input width D it accepts (1 <= D <= 768): the input width picks the layer-0 code path -- the
fused layer kernels' specialisations (nk = ceil(D / 16) in {4, 5, 16}) or their generic run-time-nk instantiation, an x ring of
12, 6, 4 or 3 stages (8 KB x ceil(D / 64) per stage), and above 256 the K-split projection in 256-wide chunks, the last one
possibly partial.  Each width is held to the oracle, and to the same model zero-padded to a width whose kernel other tests hold
to the oracle, bit for bit.  Also: every projection variant on the K-split path, the refusal of D > 768, and packers that
write every byte the kernels read.  Run on the B200 box: pytest -m gpu."""
import pytest
import torch

import util

pytestmark = pytest.mark.gpu

B, T, L = 37, 33, 2
WIDTHS = [1, 8,                  # nk = 1; D < 8 splits its input through split_planes_pad
          17, 33, 48,            # generic kernel, D % 8 != 0
          63, 64, 65, 72,        # nk = 4 / 5 specialisations with partial k-steps; 64 = one whole k-block
          100, 128,              # generic kernel, 6-stage ring
          129, 160, 192,         # 4-stage ring
          193, 200, 240,         # generic kernel, 3-stage ring
          241, 255,              # nk = 16 with a partial k-step
          257, 300, 512, 513, 700, 767]   # K-split layer 0: partial and whole last chunks


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import b200vad  # noqa: F401
    return torch.device("cuda:0")


def _input(D, seed):
    return torch.randn(B, T, D, generator=torch.Generator().manual_seed(seed))


def _oracle(D, x, sigma, layers=L):
    return util.make_oracle("PyanNet2", {"encoding_dim": D, "lstm": {"hidden_size": 128, "num_layers": layers, "bidirectional": True,
                                                                     "monolithic": True, "dropout": 0.0}},
                            spread=True, feats=x, sigma=sigma)


def _run(blob, x, mode, kernel=2, terms=2, layers=L):
    """Probabilities of lstm_head under LSTM mode / projection kernel / projection terms; the caller restores the defaults."""
    import b200vad
    lib = b200vad.lib()
    b200vad._lib.check(lib.b200vad_set_lstm_fused(mode), "set_lstm_fused")
    b200vad._lib.check(lib.b200vad_set_projection_kernel(kernel), "set_projection_kernel")
    b200vad._lib.check(lib.b200vad_set_projection_terms(terms), "set_projection_terms")
    return torch.ops.b200vad.lstm_head(x, blob, layers).cpu()


def _restore_defaults():
    import b200vad
    lib = b200vad.lib()
    lib.b200vad_set_lstm_fused(1)
    lib.b200vad_set_projection_kernel(2)
    lib.b200vad_set_projection_terms(2)


@pytest.mark.parametrize("D", WIDTHS)
def test_width_against_oracle(dev, D):
    """Modes 1 and 2 (fused layer kernels) at trained-model logit spread: within PROB_RTOL of the oracle and bit-identical to
    each other.  Mode 0 keeps a single-plane W_hh on every layer and is held to the oracle at sigma = 0.5 elsewhere."""
    import b200vad
    x = _input(D, D)
    o = _oracle(D, x, 2.0)
    with torch.no_grad():
        ref = o(x).squeeze(-1)
    blob = b200vad.pack_model(o.model.state_dict(), dev, D, L)
    try:
        out = {mode: _run(blob, x.to(dev), mode) for mode in (1, 2)}
    finally:
        _restore_defaults()
    err = util.prob_err(out[1], ref)
    print(f"D={D}: rel err of p vs oracle {err:.2e}")
    assert torch.equal(out[1], out[2]), f"D={D}: mode 1 != mode 2"
    assert err <= util.PROB_RTOL, (D, err)


@pytest.mark.parametrize("D", WIDTHS)
def test_zero_padded_width_is_bit_identical(dev, D):
    """lstm_head at width D equals lstm_head at width Dp (256 below 256: the nk = 16 kernel; 768 above: three whole K chunks)
    with zero input channels and random weight columns appended, bit for bit, in every LSTM mode.  The padded channels split
    to hi = lo = 0, both runs align their k-steps to 16, and K chunks past the data add exact zeros into xg."""
    import b200vad
    Dp = 256 if D < 256 else 768
    x = _input(D, D)
    o = _oracle(D, x, 2.0)
    sd = o.model.state_dict()
    sdp, xp = util.pad_input_width(sd, x, Dp, seed=D)
    blob = b200vad.pack_model(sd, dev, D, L)
    blob_p = b200vad.pack_model(sdp, dev, Dp, L)
    try:
        for mode in (0, 1, 2):
            a = _run(blob, x.to(dev), mode)
            b = _run(blob_p, xp.to(dev), mode)
            assert torch.isfinite(a).all(), (D, mode)
            assert torch.equal(a, b), f"D={D} -> {Dp}, mode {mode}: max |diff| {(a - b).abs().max().item():.3e}"
    finally:
        _restore_defaults()


@pytest.mark.parametrize("D", [300, 768])
def test_projection_variants_on_the_k_split_path(dev, D):
    """Layer 0 runs on the K-split kernel whatever the projection kernel when D > 256.  Modes 1 and 2: the fused layer 1 takes
    2 products (terms 2) or 3 (terms 3) whatever the projection kernel, so all three kernels give the same bits.  Mode 0:
    layer 1 runs on the projection kernel; kernels 1 and 2 agree bit for bit at equal terms, and kernel 0 (always 3 products)
    equals both at terms 3.  Terms 2 and 3 agree within 1e-4.  Modes 1 and 2 are held to the oracle at sigma = 2, mode 0
    (single-plane W_hh) at sigma = 0.5."""
    import b200vad
    x = _input(D, 5 * D)
    models = {}
    for sigma in (2.0, 0.5):
        o = _oracle(D, x, sigma)
        with torch.no_grad():
            models[sigma] = (b200vad.pack_model(o.model.state_dict(), dev, D, L), o(x).squeeze(-1))
    xd = x.to(dev)
    out = {}
    try:
        for mode in (0, 1, 2):
            blob, _ = models[0.5 if mode == 0 else 2.0]
            for kernel in (0, 1, 2):
                for terms in (2, 3):
                    out[(mode, kernel, terms)] = _run(blob, xd, mode, kernel, terms)
    finally:
        _restore_defaults()
    for (mode, kernel, terms), p in out.items():
        err = util.prob_err(p, models[0.5 if mode == 0 else 2.0][1])
        print(f"D={D} mode {mode} kernel {kernel} terms {terms}: rel err of p vs oracle {err:.2e}")
    for mode in (1, 2):
        for terms in (2, 3):
            for kernel in (0, 1):
                assert torch.equal(out[(mode, kernel, terms)], out[(mode, 2, terms)]), \
                    f"D={D} mode {mode} terms {terms}: projection kernel {kernel} != kernel 2"
            assert torch.equal(out[(1, 2, terms)], out[(2, 2, terms)]), f"D={D} terms {terms}: mode 1 != mode 2"
    for terms in (2, 3):
        assert torch.equal(out[(0, 1, terms)], out[(0, 2, terms)]), f"D={D} mode 0 terms {terms}: kernel 1 != kernel 2"
    assert torch.equal(out[(0, 0, 3)], out[(0, 2, 3)]), f"D={D} mode 0 terms 3: kernel 0 != kernel 2"
    for mode in (0, 1, 2):
        for kernel in (0, 1, 2):
            assert util.prob_err(out[(mode, kernel, 2)], out[(mode, kernel, 3)]) <= 1e-4, (D, mode, kernel)
    for (mode, kernel, terms), p in out.items():
        assert util.prob_err(p, models[0.5 if mode == 0 else 2.0][1]) <= util.PROB_RTOL, (D, mode, kernel, terms)


def test_inputs_wider_than_768_are_refused(dev):
    """b200vad_model_workspace_bytes sizes for D <= 768; a wider input is refused at packing and at the forward call with
    B200VAD_EINVAL at every batch size -- not accepted at large B and "workspace too small" at small B."""
    import b200vad
    import oracle
    lib = b200vad.lib()
    D, layers, Tw = 1024, 4, 50
    blob = torch.zeros(64 << 20, dtype=torch.uint8, device=dev)       # larger than any blob of this width would be
    got = {}
    for Bw in (1, 4096):
        x = torch.zeros(Bw, Tw, D, device=dev)
        prob = torch.empty(Bw, Tw, device=dev)
        ws = torch.empty(lib.b200vad_model_workspace_bytes(Bw, Tw), dtype=torch.uint8, device=dev)
        rc = lib.b200vad_model_forward_f32(blob.data_ptr(), D, layers, x.data_ptr(), Bw, Tw, prob.data_ptr(), ws.data_ptr(),
                                           ws.numel(), torch.cuda.current_stream(dev).cuda_stream)
        torch.cuda.synchronize()
        got[Bw] = (rc, lib.b200vad_last_error().decode() if rc else "")
    assert all(rc == -1 and "768" in msg for rc, msg in got.values()), got       # B200VAD_EINVAL
    assert lib.b200vad_model_packed_bytes(D, layers) == 0
    torch.manual_seed(0)
    o = oracle.VadModel("PyanNet2", {"encoding_dim": D}).eval()
    with pytest.raises(b200vad.B200VadError, match="768"):
        b200vad.pack_model(o.model.state_dict(), dev, D, layers)


def _pack_model_into(blob, sd, dev, D, layers):
    """b200vad_model_pack_* on a caller-allocated buffer, as a C caller does it."""
    import b200vad
    from b200vad.packing import lstm_param
    lib = b200vad.lib()
    st = torch.cuda.current_stream(dev).cuda_stream
    keep = []
    for layer in range(layers):
        for d in (0, 1):
            ws = [lstm_param(sd, "", n, layer, d == 1, True).float().contiguous().to(dev)
                  for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]
            keep += ws
            b200vad._lib.check(lib.b200vad_model_pack_lstm(blob.data_ptr(), D, layers, layer, d, *[w.data_ptr() for w in ws], st),
                               "b200vad_model_pack_lstm")
    hs = [sd[k].float().contiguous().to(dev) for k in ("linear.0.weight", "linear.0.bias", "linear.1.weight", "linear.1.bias",
                                                       "classifier.weight", "classifier.bias")]
    b200vad._lib.check(lib.b200vad_model_pack_head(blob.data_ptr(), D, layers, *[h.data_ptr() for h in hs], st),
                       "b200vad_model_pack_head")
    torch.cuda.synchronize()


@pytest.mark.parametrize("D", [60, 100, 256, 300])
@pytest.mark.parametrize("layers", [1, 4])
def test_model_packer_writes_every_byte_read(dev, D, layers):
    """pack_model packs into a zeroed buffer, which would hide a byte the C packers leave unwritten; a C caller's cudaMalloc
    buffer holds anything.  Packed into a buffer of 0xFF bytes (fp16 NaN), the model must give the same bits in every mode."""
    import b200vad
    x = _input(D, D + layers)
    o = _oracle(D, x, 2.0, layers)
    sd = o.model.state_dict()
    ref_blob = b200vad.pack_model(sd, dev, D, layers)
    blob = torch.full_like(ref_blob, 0xFF)
    _pack_model_into(blob, sd, dev, D, layers)
    try:
        for mode in (0, 1, 2):
            a = _run(blob, x.to(dev), mode, layers=layers)
            assert torch.equal(a, _run(ref_blob, x.to(dev), mode, layers=layers)), (D, layers, mode)
    finally:
        _restore_defaults()


def test_sincnet_packer_writes_every_byte_read(dev):
    """The same for b200vad_sincnet_pack: SincNet features from a blob packed into 0xFF bytes equal those from a zeroed blob."""
    import b200vad
    from b200vad.packing import SINCNET_KEYS
    lib = b200vad.lib()
    o = util.make_oracle("PyanNet", {})
    sd = o.model.state_dict()
    ref_blob = b200vad.pack_sincnet(sd, dev)
    blob = torch.full_like(ref_blob, 0xFF)
    ts = [sd["sincnet." + k].float().contiguous().to(dev) for k in SINCNET_KEYS]
    b200vad._lib.check(lib.b200vad_sincnet_pack(blob.data_ptr(), *[t.data_ptr() for t in ts],
                                                 torch.cuda.current_stream(dev).cuda_stream), "b200vad_sincnet_pack")
    torch.cuda.synchronize()
    wav = util.synth_wave(3, 16000 + 1234, seed=2).to(dev)
    a = torch.ops.b200vad.sincnet(wav, blob)
    assert torch.isfinite(a).all()
    assert torch.equal(a, torch.ops.b200vad.sincnet(wav, ref_blob))
