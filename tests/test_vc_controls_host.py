"""Per-request seeds and controls of per-item synthesizer batches, without a GPU: the Philox4x32-10 model against the
Random123 known answers, and the argument checks (they all run before any kernel launch)."""
import numpy as np
import pytest
import torch

import megatts2_hierspeechpp_b200 as hsv
from megatts2_hierspeechpp_b200 import ops
from megatts2_hierspeechpp_b200.runtime import to_pcm16
from philox_model import philox4x32_10, seeded_normal, unit_open

B, T, TM = 3, 40, 30


@pytest.mark.parametrize("ctr,key,want", [
    ([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
    ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
    ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0],
     [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]),
])
def test_philox_known_answers(ctr, key, want):
    assert philox4x32_10(np.array(ctr, np.uint64), np.array(key, np.uint64)).tolist() == want


def test_uniforms_lie_strictly_inside_the_unit_interval():
    u = unit_open(np.array([0, 1, 255, 256, 0x7fffffff, 0xffffff00, 0xffffffff], np.uint32))
    assert u.dtype == np.float32 and (u > 0).all() and (u < 1).all()
    assert u[0] == np.float32(2.0 ** -24) and u[-1] == np.float32(1 - 2.0 ** -24)


def test_model_depends_on_seed_channel_and_frame_only():
    a = seeded_normal(7, 3, 13)
    assert np.array_equal(a[:, :9], seeded_normal(7, 3, 9)) and np.array_equal(a[:2], seeded_normal(7, 2, 13))
    assert not np.array_equal(a, seeded_normal(8, 3, 13))
    assert np.array_equal(seeded_normal(-1, 2, 5), seeded_normal((1 << 64) - 1, 2, 5))      # int64 seeds as 64 bits
    assert np.abs(a).max() <= np.sqrt(48 * np.log(2)) + 1e-12


# ---------------------------------------------------------------------------------------------- argument checks
@pytest.fixture(scope="module")
def model():
    return hsv.HierSpeechSynthesizer().eval()


def _args(pairs=True, **over):
    a = dict(src=torch.zeros(B, 1024, T), src_length=[40, 17, 1], trg_mel=torch.zeros((2 if pairs else 1) * B, 80, TM),
             trg_length=[30, 9, 30] * (2 if pairs else 1), f0=torch.zeros(B, 1, 4 * T))
    a.update(over)
    return a


def _vcnc(model, per_item=True, noise_scale=0.333, denoise_ratio=0.3, **kw):
    a = _args()
    return model.voice_conversion_noise_control(a["src"], a["src_length"], a["trg_mel"], a["trg_length"], a["f0"],
                                                noise_scale, False, denoise_ratio, per_item=per_item, **kw)


def _vc(model, per_item=True, noise_scale=0.333, **kw):
    a = _args(pairs=False)
    return model.voice_conversion(a["src"], a["src_length"], a["trg_mel"], a["trg_length"], a["f0"], noise_scale,
                                  per_item=per_item, **kw)


def _infer(model, per_item=True, **kw):
    a = _args()
    return model.infer(torch.zeros(B, 80, T), a["src"], a["src_length"], a["f0"], per_item=per_item, **kw)


SEEDS = [1, 2, 3]


@pytest.mark.parametrize("call", [_vcnc, _vc, _infer])
@pytest.mark.parametrize("bad", [
    dict(seed=SEEDS, eps=torch.zeros(B, 192, T)),                           # seed and eps together
    dict(seed=SEEDS, per_item=False),
    dict(seed=[1, 2]),                                                      # one seed per item
    dict(seed=torch.tensor([1, 2, 3], dtype=torch.int32)),                  # wrong dtype
    dict(seed=torch.tensor([[1, 2, 3]])),                                   # wrong shape
    dict(seed=torch.tensor([1, 2, 3], device="meta")),                      # wrong device
    dict(seed=[1, 2, 1 << 63]),                                             # past int64
    dict(seed=5),                                                           # not one per item
    dict(seed=[1, 2.5, 3]),                                                 # not an integer
    dict(seed=__import__("numpy").int64(5)),                                # a lone numpy integer
])
def test_seed_argument_checks(model, call, bad):
    with pytest.raises(ValueError):
        call(model, **bad)


@pytest.mark.parametrize("call", [_vcnc, _vc])
@pytest.mark.parametrize("bad", [
    dict(noise_scale=torch.full((B,), 0.5), per_item=False),
    dict(noise_scale=torch.full((B - 1,), 0.5)),
    dict(noise_scale=torch.full((B, 1), 0.5)),
    dict(noise_scale=torch.ones(B, dtype=torch.int64)),
    dict(noise_scale=torch.full((B,), 0.5, device="meta")),
])
def test_noise_scale_argument_checks(model, call, bad):
    with pytest.raises(ValueError):
        call(model, **bad)


@pytest.mark.parametrize("bad", [
    dict(denoise_ratio=torch.full((B,), 0.5), per_item=False),
    dict(denoise_ratio=torch.full((2 * B,), 0.5)),
    dict(denoise_ratio=torch.zeros(B, dtype=torch.int32)),
])
def test_denoise_ratio_argument_checks(model, bad):
    with pytest.raises(ValueError):
        _vcnc(model, **bad)


@pytest.mark.parametrize("call", [_vcnc, _vc, _infer])
def test_valid_controls_pass_the_checks(model, call):
    # the checks pass; the call then stops at the first kernel input (CUDA tensors only, no CPU fallback)
    kw = dict(seed=torch.tensor(SEEDS))
    if call is not _infer:
        kw["noise_scale"] = torch.rand(B, dtype=torch.float64)
    if call is _vcnc:
        kw["denoise_ratio"] = torch.rand(B)
    with pytest.raises(RuntimeError, match="CUDA"):
        call(model, **kw)


def test_posterior_encoder_seed_needs_lengths(model):
    x, f0 = torch.zeros(B, 1024, T), torch.zeros(B, 1, 4 * T)
    with pytest.raises(ValueError):
        model.enc_p_l(x, f0, None, seed=SEEDS)
    with pytest.raises(ValueError):
        model.enc_p_l(x, f0, None, noise_scale=torch.ones(B))
    with pytest.raises(ValueError):
        model.enc_p_l(x, f0, None, lengths=[40, 17, 1], seed=SEEDS, eps=torch.zeros(B, 192, T))


def test_pcm_per_row_scale_argument_checks():
    audio, p = torch.zeros(B, 100), torch.ones(B)
    for kw in (dict(per_utterance=False), dict(scale_norm="max", per_utterance=True),
               dict(order="speechsr", per_utterance=True)):
        with pytest.raises(ValueError):
            to_pcm16(audio, **{"scale_norm": "prompt", **kw}, prompt_audio_max=p)
    for bad in (torch.ones(B + 1), torch.ones(B, 1), torch.ones(B, dtype=torch.int32)):
        with pytest.raises(ValueError):
            to_pcm16(audio, "prompt", bad, per_utterance=True)
    with pytest.raises(RuntimeError, match="CUDA"):
        to_pcm16(audio, "prompt", p, per_utterance=True)


def test_noise_ops_refuse_cpu_tensors():
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.seeded_normal(torch.tensor([1]), 4, 8)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.sample_ragged(torch.zeros(1, 8, 8), 1.0, seeds=torch.tensor([1]))


@pytest.mark.parametrize("per_item", [False, True])
@pytest.mark.parametrize("scalar", [torch.tensor(0.5), torch.tensor([0.5]), torch.tensor(1)])
def test_one_element_control_tensors_stay_scalars(model, per_item, scalar):
    # as before per-item controls existed: one value for the whole call; the checks pass and the call then stops at the
    # first kernel input (CUDA tensors only)
    ln = torch.tensor([40, 17, 1])                 # per_item=False takes the reference's length tensors
    a, v = _args(src_length=ln, trg_length=torch.tensor([30, 9, 30] * 2)), _args(False, src_length=ln,
                                                                              trg_length=torch.tensor([30, 9, 30]))
    with pytest.raises(RuntimeError, match="CUDA"):
        model.voice_conversion_noise_control(a["src"], a["src_length"], a["trg_mel"], a["trg_length"], a["f0"], scalar,
                                             False, scalar, per_item=per_item)
    with pytest.raises(RuntimeError, match="CUDA"):
        model.voice_conversion(v["src"], v["src_length"], v["trg_mel"], v["trg_length"], v["f0"], scalar,
                               per_item=per_item)
