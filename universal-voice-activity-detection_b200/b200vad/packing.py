"""Pack reference-layout state dicts (torch fp32 parameters) into the kernels' device layout.

State-dict keys are those of the reference modules: ``lstm.{weight_ih,weight_hh,bias_ih,bias_hh}_l{k}[_reverse]``
(nn.LSTM, PyanNet2.py:95) or ``lstm.{k}.*_l0[_reverse]`` (monolithic=False, PyanNet2.py:98-120),
``linear.{0,1}.{weight,bias}``, ``classifier.{weight,bias}``; SincNet: ``wav_norm1d.*``,
``conv1d.0.filterbank.{low_hz_,band_hz_,window_,n_}``, ``conv1d.{1,2}.*``, ``norm1d.{0,1,2}.*`` (sincnet.py:44-71).
"""

from __future__ import annotations

import torch

from . import _lib


def _f32(t: torch.Tensor, device) -> torch.Tensor:
    return t.detach().to(device=device, dtype=torch.float32).contiguous()


def _stream(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def lstm_param(sd: dict, prefix: str, name: str, layer: int, reverse: bool, monolithic: bool) -> torch.Tensor:
    suffix = "_reverse" if reverse else ""
    if monolithic:
        return sd[f"{prefix}lstm.{name}_l{layer}{suffix}"]
    return sd[f"{prefix}lstm.{layer}.{name}_l0{suffix}"]


def pack_model(sd: dict, device, encoding_dim: int, num_layers: int = 4, monolithic: bool = True, prefix: str = "") -> torch.Tensor:
    """LSTM stack + linear head -> opaque uint8 device blob for b200vad::lstm_head."""
    device = torch.device(device)
    if device.type != "cuda":
        raise _lib.B200VadError("packing needs a CUDA device (no CPU path)")
    L = _lib.lib()
    for key in ("linear.0.weight", "linear.1.weight", "classifier.weight"):
        if prefix + key not in sd:
            raise _lib.B200VadError(f"state dict lacks {prefix + key}: only linear.num_layers == 2 is supported by the fused head")
    nbytes = L.b200vad_model_packed_bytes(encoding_dim, num_layers)
    blob = torch.zeros(nbytes, dtype=torch.uint8, device=device)
    keep = []
    with torch.cuda.device(device):
        st = _stream(device)
        for layer in range(num_layers):
            for d in (0, 1):
                ws = [_f32(lstm_param(sd, prefix, n, layer, d == 1, monolithic), device)
                      for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]
                D_l = encoding_dim if layer == 0 else 256
                if tuple(ws[0].shape) != (512, D_l) or tuple(ws[1].shape) != (512, 128):
                    raise _lib.B200VadError(
                        f"unsupported LSTM shape {tuple(ws[0].shape)}/{tuple(ws[1].shape)}: the kernels are built for "
                        "hidden_size=128, bidirectional=True (the reference defaults)")
                keep += ws
                _lib.check(L.b200vad_model_pack_lstm(blob.data_ptr(), encoding_dim, num_layers, layer, d,
                                                     ws[0].data_ptr(), ws[1].data_ptr(), ws[2].data_ptr(), ws[3].data_ptr(), st),
                           "b200vad_model_pack_lstm")
        hs = [_f32(sd[prefix + k], device) for k in ("linear.0.weight", "linear.0.bias", "linear.1.weight", "linear.1.bias",
                                                     "classifier.weight", "classifier.bias")]
        if tuple(hs[0].shape) != (128, 256) or tuple(hs[2].shape) != (128, 128) or hs[4].numel() != 128:
            raise _lib.B200VadError("unsupported head shape: expected Linear(256,128), Linear(128,128), Linear(128,1)")
        keep += hs
        _lib.check(L.b200vad_model_pack_head(blob.data_ptr(), encoding_dim, num_layers, *[h.data_ptr() for h in hs], st),
                   "b200vad_model_pack_head")
        torch.cuda.current_stream(device).synchronize()   # sources may be temporaries
    return blob


# SincNet parameters in the argument order of b200vad_sincnet_pack
SINCNET_KEYS = ("wav_norm1d.weight", "wav_norm1d.bias", "conv1d.0.filterbank.low_hz_", "conv1d.0.filterbank.band_hz_",
                "conv1d.0.filterbank.window_", "conv1d.0.filterbank.n_", "conv1d.1.weight", "conv1d.1.bias",
                "conv1d.2.weight", "conv1d.2.bias", "norm1d.0.weight", "norm1d.0.bias", "norm1d.1.weight", "norm1d.1.bias",
                "norm1d.2.weight", "norm1d.2.bias")


def pack_sincnet(sd: dict, device, prefix: str = "sincnet.") -> torch.Tensor:
    device = torch.device(device)
    if device.type != "cuda":
        raise _lib.B200VadError("packing needs a CUDA device (no CPU path)")
    L = _lib.lib()
    ts = [_f32(sd[prefix + k], device) for k in SINCNET_KEYS]
    if tuple(ts[6].shape) != (60, 80, 5) or tuple(ts[8].shape) != (60, 60, 5) or ts[2].numel() != 40 or ts[4].numel() != 125:
        raise _lib.B200VadError("unsupported SincNet shape (expected the reference's 80x251 sinc + 60x80x5 + 60x60x5)")
    blob = torch.zeros(L.b200vad_sincnet_packed_bytes(), dtype=torch.uint8, device=device)
    with torch.cuda.device(device):
        _lib.check(L.b200vad_sincnet_pack(blob.data_ptr(), *[t.data_ptr() for t in ts], _stream(device)), "b200vad_sincnet_pack")
        torch.cuda.current_stream(device).synchronize()
    return blob
