"""Per-item batches of the text-to-vec tail without a GPU: the ``lengths=`` argument checks of ``W2VDecoder``,
``PitchPredictor`` and ``TTVTail`` all run before any kernel launch."""
import pytest
import torch

import megatts2_hierspeechpp_b200 as hsv

B, T = 3, 40


@pytest.fixture(scope="module")
def tail():
    return hsv.TTVTail().eval()


def _calls(tail, lengths):
    z, g = torch.zeros(B, 256, T), torch.zeros(B, 256, 1)
    w2v = torch.zeros(B, 1024, T)
    return [lambda: tail(z, None, g, lengths=lengths),
            lambda: tail(z, torch.ones(B, 1, T), g, lengths=lengths),
            lambda: tail.w2v_decoder(z, None, g=g, lengths=lengths),
            lambda: tail.pp(w2v, g, lengths=lengths)]


@pytest.mark.parametrize("bad", [
    [40, 17],                                              # one length per item
    [41, 17, 1],                                           # past T
    [40, 0, 1],                                            # empty item
    [40, 17, -3],
    torch.tensor([[40, 17, 1]]),                           # wrong shape
    torch.tensor([40.0, 17.0, 1.0]),                       # wrong dtype
    torch.tensor([40, 17, 1], dtype=torch.int16),
    torch.tensor([40, 17, 1], device="meta"),              # wrong device
], ids=["count", "past-T", "zero", "negative", "shape", "float", "int16", "device"])
def test_lengths_argument_checks(tail, bad):
    for call in _calls(tail, bad):
        with pytest.raises(ValueError):
            call()


@pytest.mark.parametrize("good", [[40, 17, 1], torch.tensor([40, 17, 1]), torch.tensor([40, 17, 1], dtype=torch.int32)],
                         ids=["host", "int64", "int32"])
def test_valid_lengths_pass_the_checks(tail, good):
    # the checks pass; the call then stops at the first kernel input (CUDA tensors only, no CPU fallback)
    for call in _calls(tail, good):
        with pytest.raises(RuntimeError, match="CUDA"):
            call()


def test_resblock_masked_forward_still_raises(tail):
    with pytest.raises(NotImplementedError):
        tail.pp.resblocks[0](torch.zeros(1, 128, 8), torch.ones(1, 1, 8))
