"""Per-request seeds and controls of per-item synthesizer batches on the GPU.

The seeded noise (csrc/noise.cu) against its numpy model and as a distribution; its independence of the batch; the
fused sampling launch against ``frame_op(OP_SAMPLE)`` fed with the same noise; each of the three per-item calls with
per-item seeds, noise scales and denoise ratios against the batch-1 call of every item; one captured graph for every
mix; and the per-row PCM scale."""
import numpy as np
import pytest
import torch

from philox_model import seeded_normal as model_normal
from test_gpu_synth_ragged import LENS, PROMPTS, _batch, _check_items, _garbage_tail, _job, _lens, synthesizer  # noqa: F401

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SEEDS = [7, -3, (1 << 62) + 1, 12345, 0]


def _seeds(vals):
    return torch.tensor(vals, dtype=torch.int64, device=DEV)


# ---------------------------------------------------------------------------------------------- the generator
# Bound of the kernel against the model's exact value of the same formula (same fp32 uniforms): logf and sincospif
# are each within 1 ulp (CUDA C Programming Guide, single-precision functions), sqrtf and the two products are
# correctly rounded (0.5 ulp each, the sqrt halving its input's relative error), so the relative error stays below
# 3 * 2^-23 and the result within 4 fp32 ulp of itself.
ULP_BOUND = 4


@pytest.mark.parametrize("C,T", [(192, 1000), (3, 4097), (1, 5)])
def test_seeded_normal_matches_the_model(hsv, C, T):
    got = hsv.ops.seeded_normal(_seeds(SEEDS), C, T).cpu().numpy()
    worst = 0.0
    for b, s in enumerate(SEEDS):
        ref = model_normal(s, C, T)
        ulp = np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64)
        worst = max(worst, float((np.abs(got[b] - ref) / ulp).max()))
    print(f"\n[seeded_normal] C={C} T={T}: max {worst:.2f} ulp from the model")
    assert worst <= ULP_BOUND


def test_seeded_normal_distribution(hsv):
    from scipy import stats
    x = hsv.ops.seeded_normal(_seeds([100, 101, 102, 103]), 256, 16384).double()      # 16.8 M samples
    n = x.numel()
    flat = x.flatten()
    m, v = flat.mean().item(), flat.var().item()
    z = (flat - m) / v ** 0.5
    skew, kurt = (z ** 3).mean().item(), (z ** 4).mean().item() - 3
    print(f"\n[seeded_normal] n={n} mean={m:.2e} var-1={v - 1:.2e} skew={skew:.2e} excess kurtosis={kurt:.2e}")
    assert abs(m) < 5 / n ** 0.5 and abs(v - 1) < 5 * (2 / n) ** 0.5
    assert abs(skew) < 5 * (6 / n) ** 0.5 and abs(kurt) < 5 * (24 / n) ** 0.5
    ks = stats.kstest(flat.cpu().numpy(), "norm")
    print(f"[seeded_normal] KS D={ks.statistic:.2e} p={ks.pvalue:.3f}")
    assert ks.pvalue > 1e-3

    def corr(a, b):
        a, b = a - a.mean(), b - b.mean()
        return ((a * b).mean() / (a.std() * b.std())).item(), a.numel()

    pairs = {"seed": (x[1:], x[:-1]), "channel": (x[:, 1:], x[:, :-1]), "frame group": (x[..., 4:], x[..., :-4]),
             "frame": (x[..., 1:], x[..., :-1]), "frame+2": (x[..., 2:], x[..., :-2])}
    for name, (a, b) in pairs.items():
        r, k = corr(a, b)
        print(f"[seeded_normal] corr({name} neighbours) = {r:.2e} (bound {5 / k ** 0.5:.2e})")
        assert abs(r) < 5 / k ** 0.5, name


def test_seeded_normal_does_not_depend_on_the_batch(hsv):
    ops = hsv.ops
    lens = [301, 150, 7]
    seeds = _seeds([11, -5, (1 << 40) + 3])
    big = ops.seeded_normal(seeds, 192, 301, valid_len=_lens(lens))
    _check_items(big, lambda b: ops.seeded_normal(seeds[b:b + 1], 192, lens[b]), lens)
    flipped = ops.seeded_normal(seeds.flip(0), 192, 257)                    # other positions, B, T, no lengths
    for b, n in enumerate(lens):
        k = min(n, 257)
        assert torch.equal(flipped[2 - b, :, :k], big[b, :, :k]), b
    assert torch.equal(ops.seeded_normal(seeds[1:2], 192, 5)[0], big[1, :, :5])
    vl = _lens(lens)
    graph = torch.cuda.CUDAGraph()
    torch.cuda.synchronize()
    with torch.cuda.graph(graph):
        captured = ops.seeded_normal(seeds, 192, 301, valid_len=vl)
    graph.replay()
    assert torch.equal(captured, big)


@pytest.mark.parametrize("noise", ["seeds", "eps"])
def test_fused_sample_equals_op_sample(hsv, noise):
    ops = hsv.ops
    lens = [203, 200, 64, 3, 1]
    B, C, T = len(lens), 192, 203
    gen = torch.Generator().manual_seed(5)
    stats = _garbage_tail(torch.randn(B, 2 * C, T, generator=gen).to(DEV), lens, seed=1)
    seeds = _seeds(SEEDS)
    vl = _lens(lens)
    eps = _garbage_tail(ops.seeded_normal(seeds, C, T), lens, seed=2)
    svec = (torch.rand(B, generator=gen) * 0.6 + 0.2).to(DEV)
    kw = {"seeds": seeds} if noise == "seeds" else {"eps": eps}

    def op_sample(b, s):
        n = lens[b]
        z = torch.empty(1, C, n, device=DEV)
        ops.frame_op(ops.OP_SAMPLE, stats[b:b + 1, :, :n].contiguous(), eps[b:b + 1, :, :n].contiguous(), None,
                     torch.ones(1, n, device=DEV), z, None, 1, C, n, s=s)
        return z

    _check_items(ops.sample_ragged(stats, svec, vl, **kw), lambda b: op_sample(b, float(svec[b])), lens)
    _check_items(ops.sample_ragged(stats, 0.333, vl, **kw), lambda b: op_sample(b, 0.333), lens)
    if noise == "seeds":                                            # no lengths: every frame
        full = ops.sample_ragged(stats[:1, :, :200].contiguous(), 0.5, seeds=seeds[:1])
        assert torch.equal(full, op_sample(0, 0.5)[:, :, :200])


# ---------------------------------------------------------------------------------------------- whole calls
def _controls(B, seed=0):
    gen = torch.Generator().manual_seed(seed)
    ns = (torch.rand(B, generator=gen) * 0.6 + 0.2).to(DEV)               # noise_scale in [0.2, 0.8]
    r = torch.rand(B, generator=gen, dtype=torch.float64).to(DEV)           # denoise_ratio in [0, 1]
    return ns, r


def _call(synthesizer, method, src, vl, mel, tl, f0, ns, r, **kw):
    if method == "voice_conversion_noise_control":
        return synthesizer.voice_conversion_noise_control(src, vl, mel, tl, f0, ns, False, r, per_item=True, **kw)
    if method == "voice_conversion":
        return synthesizer.voice_conversion(src, vl, mel, tl, f0, ns, per_item=True, **kw)
    return synthesizer.infer(mel, src, vl, f0, per_item=True, **kw)[0]


@pytest.mark.parametrize("noise", ["seed", "eps"])
@pytest.mark.parametrize("method", ["voice_conversion_noise_control", "voice_conversion", "infer"])
def test_items_with_their_own_seed_and_controls_equal_their_own_calls(hsv, synthesizer, method, noise):
    lens, prompts = LENS, PROMPTS
    if method == "infer":
        prompts = lens
    B, T, Tm = len(lens), max(lens), max(prompts)
    items = _job(lens, prompts)
    if method == "infer":
        items = [(w, f, torch.randn(1, 80, n, generator=torch.Generator().manual_seed(n)).to(DEV) * 2 - 4)
                 for (w, f, _), n in zip(items, lens)]
    pairs = method == "voice_conversion_noise_control"
    src, f0, mel = _batch(items, lens, prompts, T, Tm, pairs=pairs)
    seeds = _seeds(SEEDS)
    ns, r = _controls(B)
    vl, tl = _lens(lens), _lens(prompts + prompts if pairs else prompts)
    own_eps = [hsv.ops.seeded_normal(seeds[b:b + 1], 192, n) for b, n in enumerate(lens)]
    if noise == "seed":
        kw = {"seed": seeds}
    else:
        eps = torch.zeros(B, 192, T, device=DEV)
        for b, n in enumerate(lens):
            eps[b, :, :n] = own_eps[b][0]
        kw = {"eps": _garbage_tail(eps, lens, seed=7)}
    with torch.no_grad():
        out = _call(synthesizer, method, src, vl, mel, tl, f0, ns, r, **kw)
        assert out.shape == (B, 1, 320 * T)

        def own(b):
            n, p = lens[b], prompts[b]
            w, f, m = items[b]
            ptl = _lens([p, p] if pairs else [p])
            return _call(synthesizer, method, w, _lens([n]), m if pairs or method == "infer" else m[:1], ptl, f,
                         float(ns[b]), float(r[b]), eps=own_eps[b])

        _check_items(out, own, lens, scale=320)
        if noise == "seed" and method == "voice_conversion":                      # host sequence of seeds
            assert torch.equal(_call(synthesizer, method, src, vl, mel, tl, f0, ns, r, seed=SEEDS), out)


def test_one_graph_serves_every_seed_and_control_mix(hsv, synthesizer):
    B, T, Tm = 3, 120, 100
    items = _job([T] * B, [Tm] * B, seed=50)
    src, f0, mel = _batch(items, [T] * B, [Tm] * B, T, Tm)

    def call(s, f, m, vl, tl, seeds, ns, r):
        return synthesizer.voice_conversion_noise_control(s, vl, m, tl, f, ns, False, r, per_item=True, seed=seeds)

    runner = hsv.CudaGraphRunner(call)
    with torch.no_grad():
        for k, (lens, prompts) in enumerate((([120, 13, 77], [100, 51, 9]), ([7, 120, 119], [99, 100, 64]))):
            s, f, m = (_garbage_tail(src, lens, seed=1), _garbage_tail(f0, lens, scale=4, seed=2),
                       _garbage_tail(mel, prompts + prompts, seed=3))
            vl, tl = _lens(lens), _lens(prompts + prompts)
            seeds = _seeds([1000 * k + b for b in range(B)])
            ns, r = _controls(B, seed=k + 1)
            got = runner(s, f, m, vl, tl, seeds, ns, r).clone()
            assert torch.equal(got, call(s, f, m, vl, tl, seeds, ns, r))
            assert all(bool((got[b, :, 320 * n:] == 0).all()) for b, n in enumerate(lens))
    assert runner.captures == 1


# ---------------------------------------------------------------------------------------------- PCM
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_pcm_per_row_prompt_scale(hsv, dtype):
    from megatts2_hierspeechpp_b200.runtime import to_pcm16
    gen = torch.Generator().manual_seed(3)
    audio = (torch.randn(4, 16000, generator=gen) * torch.tensor([[0.1], [1.0], [3.0], [0.5]])).to(DEV)
    p = torch.tensor([0.5, 0.9, 1.0, 0.123456789], dtype=dtype, device=DEV)
    got = to_pcm16(audio, "prompt", p, per_utterance=True)
    assert got.dtype == torch.int16 and got.shape == audio.shape
    for b in range(4):
        assert torch.equal(got[b:b + 1], to_pcm16(audio[b:b + 1], "prompt", float(p[b]))), b
    assert torch.equal(to_pcm16(audio, "prompt", torch.full((4,), 0.7, dtype=dtype, device=DEV), per_utterance=True),
                       to_pcm16(audio, "prompt", 0.7, per_utterance=True))
