"""Shared helpers for the parity tests (seeded inputs, spread-head model, tolerances)."""
import torch

# north_star tolerances: features / probabilities within 1e-3 relative (fp32 accumulate).
# Features are compared in the log domain: |d| <= 1e-3 * max(1, |ref|)  (SURVEY 8c).
FEAT_RTOL = 1e-3
PROB_RTOL = 1e-3
NEAR_THR = 1e-3 * 0.5     # |p - 0.5| band whose decisions are reported separately


def feat_err(a, ref):
    return ((a.double() - ref.double()).abs() / ref.double().abs().clamp_min(1.0)).max().item()


def prob_err(a, ref):
    return ((a.double() - ref.double()).abs() / ref.double().abs().clamp_min(1e-12)).max().item()


def make_oracle(model_name="PyanNet2", model_dict=None, seed=42, spread=False, feats=None, sigma=0.5):
    """Reference-layout model with torch default init under manual_seed(seed).  ``spread`` rescales the
    classifier so probabilities span (0, 1) on ``feats`` (random-init outputs sit within 1e-3 of a
    constant, SURVEY 7 'hard parts'), which makes decisions / segments non-degenerate.  ``sigma`` is the
    standard deviation of the logits after rescaling: 0.5 gives p in about (0.2, 0.8); 2 and 4 are what a
    TRAINED detector looks like (p from 1e-4 to 1 - 1e-4) and are where operand rounding shows."""
    import oracle
    torch.manual_seed(seed)
    m = oracle.VadModel(model_name, dict(model_dict or {})).eval()
    if spread:
        assert feats is not None
        with torch.no_grad():
            net = m.model
            x = feats
            if model_name == "PyanNet":
                x = net.sincnet(x.unsqueeze(1)).transpose(1, 2)
            y, _ = net.lstm(x)
            for lin in net.linear:
                y = torch.nn.functional.leaky_relu(lin(y))
            z = net.classifier(y)
            mu, sd = z.mean(), z.std().clamp_min(1e-6)
            scale = sigma / sd   # logits ~ N(0, sigma)
            net.classifier.weight.mul_(scale)
            net.classifier.bias.copy_((net.classifier.bias - mu) * scale)
    return m


def synth_wave(B, N, seed=0):
    import b200vad
    return b200vad.synth.meeting_batch(B, N, seed=seed)


def pad_input_width(sd, x, Dp, seed=0):
    """The same model and input at layer-0 width Dp >= D: x gets Dp - D zero channels and weight_ih_l0[_reverse] gets
    Dp - D extra columns of RANDOM values.  Every extra product is exactly zero, so a kernel that adds them in the same order
    as the products of the first D channels must return the unpadded result bit for bit."""
    g = torch.Generator().manual_seed(seed)
    D = x.shape[-1]
    out = dict(sd)
    for k in ("lstm.weight_ih_l0", "lstm.weight_ih_l0_reverse"):
        w = sd[k]
        out[k] = torch.cat([w, torch.randn(w.shape[0], Dp - D, generator=g).to(w)], dim=1)
    return out, torch.nn.functional.pad(x, (0, Dp - D))
