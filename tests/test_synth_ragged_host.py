"""Per-item synthesizer batches without a GPU: argument checks (they all run before any kernel launch) and the
micro-batch schedule of tools/bench_synth_ragged.py."""
import pytest
import torch

import megatts2_hierspeechpp_b200 as hsv
from megatts2_hierspeechpp_b200.runtime import ragged_batches, ragged_prompt_batches

B, T, TM = 3, 40, 30


@pytest.fixture(scope="module")
def model():
    return hsv.HierSpeechSynthesizer().eval()


def _args(pairs=True, **over):
    a = dict(src=torch.zeros(B, 1024, T), src_length=[40, 17, 1], trg_mel=torch.zeros((2 if pairs else 1) * B, 80, TM),
             trg_length=[30, 9, 30] * (2 if pairs else 1), f0=torch.zeros(B, 1, 4 * T), eps=None)
    a.update(over)
    return a


def _vcnc(model, a, **kw):
    return model.voice_conversion_noise_control(a["src"], a["src_length"], a["trg_mel"], a["trg_length"], a["f0"],
                                                per_item=True, eps=a["eps"], **kw)


def _vc(model, a):
    return model.voice_conversion(a["src"], a["src_length"], a["trg_mel"], a["trg_length"], a["f0"], per_item=True,
                                  eps=a["eps"])


@pytest.mark.parametrize("bad", [
    dict(trg_mel=torch.zeros(B, 80, TM)),                                   # B rows where 2B are due
    dict(trg_mel=torch.zeros(2 * B, 81, TM)),
    dict(trg_length=[30, 9, 30]),                                           # B lengths for 2B prompts
    dict(trg_length=[30, 9, 31, 1, 1, 1]),                                  # past Tm
    dict(src_length=[40, 17]),
    dict(src_length=[41, 17, 1]),
    dict(src_length=[40, 0, 1]),
    dict(src_length=torch.tensor([[40, 17, 1]])),                           # wrong shape
    dict(src_length=torch.tensor([40.0, 17.0, 1.0])),                       # wrong dtype
    dict(src_length=torch.tensor([40, 17, 1], device="meta")),              # wrong device
    dict(f0=torch.zeros(B, 1, T)),
    dict(eps=torch.zeros(B, 192, T - 1)),
    dict(eps=torch.zeros(B, 96, T)),
    dict(eps=torch.zeros(B, 192, T, dtype=torch.float64)),
])
def test_noise_control_argument_checks(model, bad):
    with pytest.raises(ValueError):
        _vcnc(model, _args(**bad))


def test_voice_conversion_takes_one_prompt_per_item(model):
    with pytest.raises(ValueError):
        _vc(model, _args(pairs=True))                                       # 2B rows where B are due
    with pytest.raises(ValueError):
        _vc(model, _args(pairs=False, trg_length=[30, 9]))


def test_infer_prompt_shares_the_source_length(model):
    src = torch.zeros(B, 1024, T)
    with pytest.raises(ValueError):
        model.infer(torch.zeros(B, 80, T + 1), src, [40, 17, 1], torch.zeros(B, 1, 4 * T), per_item=True)
    with pytest.raises(ValueError):
        model.infer(torch.zeros(B, 80, T), src, [40, 17, 41], torch.zeros(B, 1, 4 * T), per_item=True)


def test_valid_arguments_pass_the_checks(model):
    # the checks pass; the call then stops at the first kernel input (CUDA tensors only, no CPU fallback)
    with pytest.raises(RuntimeError, match="CUDA"):
        _vcnc(model, _args(eps=torch.zeros(B, 192, T)))


def test_uncond_still_raises(model):
    with pytest.raises(NotImplementedError):
        _vcnc(model, _args(), uncond=True)
    with pytest.raises(NotImplementedError):
        model.voice_conversion(*[_args(pairs=False)[k] for k in ("src", "src_length", "trg_mel", "trg_length", "f0")],
                               uncond=True, per_item=True)


def test_eps_needs_per_item(model):
    a = _args(eps=torch.zeros(1, 192, T))
    with pytest.raises(ValueError):
        model.voice_conversion_noise_control(a["src"][:1], [T], a["trg_mel"][:2], [TM, TM], a["f0"][:1], eps=a["eps"])


def test_prompt_batches_for_the_benchmark_schedule():
    g = torch.Generator().manual_seed(1111)
    n = 128
    lens = torch.randint(100, 1001, (n,), generator=g).tolist()
    prompts = torch.randint(100, 301, (n,), generator=g).tolist()
    batches = ragged_prompt_batches(range(n), lens, prompts, 16)
    assert [(ids, T) for ids, T, _ in batches] == ragged_batches(range(n), lens, 16)
    assert sorted(i for ids, _, _ in batches for i in ids) == list(range(n))
    for ids, T, Tm in batches:
        assert len(ids) <= 16 and T % 50 == 0 and Tm % 50 == 0
        assert max(prompts[i] for i in ids) <= Tm < max(prompts[i] for i in ids) + 50
        assert max(lens[i] for i in ids) <= T < max(lens[i] for i in ids) + 50
    assert len({(len(ids), T, Tm) for ids, T, Tm in batches}) <= len(batches)
    assert ragged_prompt_batches([0, 1], [10, 60], [7, 101], 1, 50, 25) == [([1], 100, 125), ([0], 50, 25)]
    with pytest.raises(ValueError):
        ragged_prompt_batches([0], [10], [10], 1, prompt_multiple=0)
