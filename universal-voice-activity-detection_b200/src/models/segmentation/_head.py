"""LSTM stack + linear head shared by PyanNet / PyanNet2 (PyanNet2.py:60-187, PyanNet.py:66-197)."""

import torch
import torch.nn as nn

import b200vad
from src.utils.helper import merge_dict, pairwise
from .._base import Base, PackedOwner, PackedWeights


class HeadMixin(PackedOwner):
    LSTM_DEFAULTS = {"hidden_size": 128, "num_layers": 4, "bidirectional": True, "monolithic": True, "dropout": 0.5}
    LINEAR_DEFAULTS = {"hidden_size": 128, "num_layers": 2}

    def _make_head(self, lstm: dict, linear: dict, encoding_dim: int):
        self.encoding_dim = encoding_dim
        monolithic = lstm["monolithic"]
        if monolithic:
            multi_layer_lstm = dict(lstm)
            del multi_layer_lstm["monolithic"]
            self.lstm = nn.LSTM(encoding_dim, **multi_layer_lstm)
        else:
            num_layers = lstm["num_layers"]
            if num_layers > 1:
                self.dropout = nn.Dropout(p=lstm["dropout"])
            one_layer_lstm = dict(lstm)
            one_layer_lstm["num_layers"] = 1
            one_layer_lstm["dropout"] = 0.0
            del one_layer_lstm["monolithic"]
            self.lstm = nn.ModuleList([
                nn.LSTM(encoding_dim if i == 0 else lstm["hidden_size"] * (2 if lstm["bidirectional"] else 1), **one_layer_lstm)
                for i in range(num_layers)])
        self._packed = PackedWeights()
        if linear["num_layers"] < 1:
            return
        lstm_out_features = self.hparams.lstm["hidden_size"] * (2 if self.hparams.lstm["bidirectional"] else 1)
        self.linear = nn.ModuleList([
            nn.Linear(i, o) for i, o in pairwise([lstm_out_features] + [self.hparams.linear["hidden_size"]] * self.hparams.linear["num_layers"])])

    def build(self):
        if self.hparams.linear["num_layers"] > 0:
            in_features = self.hparams.linear["hidden_size"]
        else:
            in_features = self.hparams.lstm["hidden_size"] * (2 if self.hparams.lstm["bidirectional"] else 1)
        self.classifier = nn.Linear(in_features, 1)
        self.activation = nn.Sigmoid()

    def _check_supported(self):
        l, n = self.hparams.lstm, self.hparams.linear
        if l["hidden_size"] != 128 or not l["bidirectional"] or n["hidden_size"] != 128 or n["num_layers"] != 2:
            raise NotImplementedError("the sm_100a kernels are built for the reference defaults: BiLSTM(128) x L, "
                                      "Linear(128) x 2 (PyanNet2.py:60-67)")
        if not 1 <= self.encoding_dim <= b200vad._lib.MAX_INPUT_DIM:
            raise NotImplementedError(f"encoding_dim {self.encoding_dim}: the sm_100a kernels take LSTM inputs of 1 to "
                                      f"{b200vad._lib.MAX_INPUT_DIM} channels")
        if torch.is_grad_enabled() and self.training and any(p.requires_grad for p in self.parameters()):
            raise NotImplementedError("b200vad implements inference only; call .eval() / torch.no_grad()")
        if self.training and l["num_layers"] > 1 and l.get("dropout", 0.0) > 0:
            # the reference applies inter-layer dropout in train mode even under no_grad (nn.LSTM dropout / self.dropout,
            # PyanNet2.py:95-120,176-181); the kernels never do
            raise NotImplementedError("b200vad runs the eval-mode forward (no inter-layer LSTM dropout); call .eval()")

    def _head_forward(self, feats: torch.Tensor) -> torch.Tensor:
        """(B, T, D) float32 CUDA -> (B, T, 1) probabilities through torch.ops.b200vad.lstm_head."""
        self._check_supported()
        sd_owner = self
        num_layers = self.hparams.lstm["num_layers"]
        blob = self._packed.get(self, feats.device, lambda: b200vad.pack_model(
            {k: v for k, v in sd_owner.state_dict().items() if not k.startswith("sincnet.")}, feats.device,
            self.encoding_dim, num_layers, monolithic=self.hparams.lstm["monolithic"]), always=self.repack_always)
        return torch.ops.b200vad.lstm_head(feats.float(), blob, num_layers).unsqueeze(-1)


__all__ = ["HeadMixin", "Base", "merge_dict"]
