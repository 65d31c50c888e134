"""CPU checks of the LSTM input-width limit: the model workspace is sized for inputs of at most 768 channels, so wider ones are
refused where they enter -- the packed-size query and the drop-in module -- instead of failing or not depending on the batch
size (the shared library loads without a GPU)."""
import pytest
import torch

from b200vad import _lib


def test_packed_bytes_refuses_inputs_wider_than_768():
    lib = _lib.lib()
    assert _lib.MAX_INPUT_DIM == 768
    for layers in (1, 4):
        for D in (1, 60, 80, 256, 767, 768):
            assert lib.b200vad_model_packed_bytes(D, layers) > 0, D
        assert lib.b200vad_model_packed_bytes(769, layers) == 0
        assert lib.b200vad_model_packed_bytes(1024, layers) == 0
        assert lib.b200vad_model_packed_bytes(0, layers) == 0


def test_dropin_refuses_inputs_wider_than_768():
    from src.models.segmentation.PyanNet2 import PyanNet2
    with torch.no_grad():
        PyanNet2(encoding_dim=768).eval()._check_supported()
        with pytest.raises(NotImplementedError, match="1024"):
            PyanNet2(encoding_dim=1024).eval()._check_supported()
