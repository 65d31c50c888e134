"""Hand-offs of the fused LSTM layer kernel (csrc/lstm_fused.cu) at the edges of its barrier participation: the pointwise warps,
their acc_ready poller and the exchange senders meet on named barriers once per (step, part) with q < nparts and, for the
exchange, s + 1 < T, so every parts count per work item (1..8), items of unequal parts counts, a partial last part and the
shortest sequences (T = 1: no exchange at all) must give the same layer outputs as the CTA-pair kernel (mode 2), bit for bit.
D = 100 and 192 run the generic instantiation of both kernels (run-time k-step count) on 6- and 4-stage x rings, D = 80 and
256 the nk = 5 and nk = 16 specialisations on 12- and 3-stage rings.  Run on the B200 box: pytest -m gpu."""
import pytest
import torch

import util

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import b200vad  # noqa: F401
    return torch.device("cuda:0")


def _batches(clusters):
    """Batch sizes and the parts per work item the mode-1 launcher gives them (B = 16 x parts; items per direction chosen from
    the step-time table): with h = clusters // 2 items per direction in one wave, B = 16 n h runs items of n parts (odd n with
    a partial last part); 16 (8 h - 1) - 5 runs two waves of 8-part items and one 7-part item with a partial last part; 5 and
    16 run one part."""
    h = max(1, clusters // 2)
    bs = [5, 16] + [16 * n * h - 5 * (n & 1) for n in range(1, 9)] + [16 * (16 * h - 1) - 5]
    return sorted(set(bs))


@pytest.mark.parametrize("D", [80, 100, 192, 256])
@pytest.mark.parametrize("T", [1, 2, 3, 50])
def test_fused_layer_equals_pair_kernel_at_every_parts_count(dev, D, T):
    import b200vad
    import oracle
    lib = b200vad.lib()
    L = 2                                          # layer 0 takes (hi, lo) planes, layer 1 the scaled split of layer 0's output
    torch.manual_seed(7)
    m = oracle.VadModel("PyanNet2", {"encoding_dim": D, "lstm": {"hidden_size": 128, "num_layers": L, "bidirectional": True,
                                                                 "monolithic": True, "dropout": 0.0}}).eval()
    blob = b200vad.pack_model(m.model.state_dict(), dev, D, L)
    # at one T, narrower inputs also run zero-padded to 256 (random weight columns): the nk = 16 kernel must give the same bits
    padded = T == 3 and D < 256
    if padded:
        sdp, _ = util.pad_input_width(m.model.state_dict(), torch.zeros(1, 1, D), 256, seed=D)
        blob_p = b200vad.pack_model(sdp, dev, 256, L)
    g = torch.Generator(device=dev).manual_seed(1000 * D + T)
    try:
        for B in _batches(lib.b200vad_lstm_fused_clusters()):
            x = torch.randn(B, T, D, device=dev, generator=g)
            if D == 80:
                x = x * 3 - 5
            out = {}
            for mode in (1, 2):
                lib.b200vad_set_lstm_fused(mode)
                out[mode] = torch.ops.b200vad.lstm_head(x, blob, L)
            if padded:
                out["pad"] = torch.ops.b200vad.lstm_head(torch.nn.functional.pad(x, (0, 256 - D)), blob_p, L)
            torch.cuda.synchronize()
            assert torch.equal(out[1], out[2]), f"B={B} T={T} D={D}: mode 1 != mode 2"
            if padded:
                assert torch.equal(out[2], out["pad"]), f"B={B} T={T} D={D}: != the same input zero-padded to 256"
    finally:
        lib.b200vad_set_lstm_fused(1)
