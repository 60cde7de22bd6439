"""Any-rate SpeechSR input on the GPU: the ragged sinc resampler (``hsv.Resample``, csrc/resample.cu) against the fp64
oracle of the same fp32 table and against torchaudio's own fp32 error, int16 and identity inputs, per-item bit
identity in padded mixed-rate batches, and ``hsv.SpeechSRAudio`` with the bundled SpeechSR checkpoints: each item
equal to its own chain, the torchaudio -> SpeechSR chain within the parity bar, and one CUDA graph for every mix."""
import math
import warnings

import numpy as np
import pytest
import torch

from conftest import MAX_ABS_TOL, SNR_DB_MIN, golden_sd
from oracle import closed_form as CF
from oracle.resample import resample_fp64

from megatts2_hierspeechpp_b200 import resample as RS

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PAIRS = [(r, 16000) for r in RS.DEFAULT_RATES if r != 16000] + [(48000, 44100)]


def _lengths(orig, new):
    o, n, width = RS.ratio(orig, new)
    return sorted({L for L in (1, 2, width - 1, o, o + 1, 3 * orig + 17, 10 * orig) if L >= 1})


def _signal(L, seed, int16):
    g = torch.Generator().manual_seed(seed)
    if int16:
        s = torch.randint(-32768, 32768, (L,), generator=g, dtype=torch.int32).to(torch.int16)
        return s, s.float() / 32768.0
    x = torch.rand(L, generator=g) * 2 - 1
    return x, x


def _torchaudio_resample(x, orig, new):
    ta = pytest.importorskip("torchaudio")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return ta.functional.resample(x, orig, new, resampling_method="kaiser_window")


@pytest.mark.parametrize("int16", [False, True], ids=["fp32", "int16"])
@pytest.mark.parametrize("orig,new", PAIRS)
def test_against_fp64(hsv, orig, new, int16):
    m = hsv.Resample((orig,), new).to(DEV)
    tab, width = RS.sinc_kaiser_table(orig, new)
    o, n, _ = RS.ratio(orig, new)
    K = tab.shape[1]
    Ls = _lengths(orig, new)
    T = max(Ls)
    xs = [_signal(L, 1000 * i + orig, int16) for i, L in enumerate(Ls)]
    x = torch.full((len(Ls), T), -7 if int16 else float("nan"), dtype=torch.int16 if int16 else torch.float32)
    for i, (raw, _) in enumerate(xs):
        x[i, :Ls[i]] = raw
    y, n_out = m(x.to(DEV), [orig] * len(Ls), Ls)
    y, n_out = y.cpu(), n_out.cpu()
    assert n_out.tolist() == m.output_lengths([orig] * len(Ls), Ls)
    err_k = err_ta = 0.0
    for i, (L, (_, xf)) in enumerate(zip(Ls, xs)):
        nb = int(n_out[i])
        y64, mag = resample_fp64(xf.numpy(), tab.numpy(), o, n, width, nb)
        d = np.abs(y[i, :nb].double().numpy() - y64)
        assert np.all(d <= K * 2.0 ** -24 * mag), (L, d.max())
        assert not y[i, nb:].any()
        err_k = max(err_k, float(d.max()))
        y_ta = _torchaudio_resample(xf, orig, new).double().numpy()
        assert y_ta.shape == (nb,)
        err_ta = max(err_ta, float(np.abs(y_ta - y64).max()))
    print(f"{orig} -> {new} {'int16' if int16 else 'fp32'}: max |y - y64| kernel {err_k:.3e}, torchaudio CPU "
          f"{err_ta:.3e}")
    assert err_k <= 2 * err_ta


def test_int16_equals_float_and_identity(hsv):
    m = hsv.Resample().to(DEV)
    rates = [16000, 44100, 48000, 16000, 8000, 22050]
    Ls = [16000, 44100 * 2 + 5, 48000, 777, 8000 * 3, 22050]
    T = max(Ls)
    s = torch.randint(-32768, 32768, (len(rates), T), generator=torch.Generator().manual_seed(5),
                      dtype=torch.int32).to(torch.int16).to(DEV)
    xf = s.float() / 32768.0
    y16, n16 = m(s, rates, Ls)
    yf, nf = m(xf, rates, Ls)
    assert torch.equal(y16, yf) and torch.equal(n16, nf)
    for b, (r, L) in enumerate(zip(rates, Ls)):
        if r == 16000:
            assert int(nf[b]) == L and torch.equal(yf[b, :L], xf[b, :L]) and not yf[b, L:].any()
    # fp32 identity keeps every bit, -0.0 and subnormals included
    special = torch.tensor([[-0.0, 1e-40, -3.5, 0.0, float("inf")]], device=DEV)
    y, n_out = m(special, [16000], [5])
    assert int(n_out[0]) == 5 and torch.equal(y.view(torch.int32), special.view(torch.int32))


def test_per_item_bit_identical(hsv):
    m = hsv.Resample().to(DEV)
    rng = np.random.default_rng(11)
    rates = [int(r) for r in rng.permutation(list(RS.DEFAULT_RATES) * 2)]
    Ls = [int(rng.integers(1, 2 * r)) for r in rates]
    Ls[0], Ls[1] = 1, 2
    T = max(Ls) + 37
    x = torch.empty(len(rates), T)
    for b, L in enumerate(Ls):
        x[b] = float("nan") if b % 2 else 1e30
        x[b, :L] = torch.rand(L, generator=torch.Generator().manual_seed(b)) * 2 - 1
    x = x.to(DEV)
    rate_t = torch.tensor(rates, dtype=torch.int32, device=DEV)
    len_t = torch.tensor(Ls, dtype=torch.int64, device=DEV)
    y, n_out = m(x, rate_t, len_t)
    assert y.shape == (len(rates), -(-16000 * T // 8000))
    assert n_out.cpu().tolist() == m.output_lengths(rates, Ls)
    for b, (r, L) in enumerate(zip(rates, Ls)):
        y1, n1 = m(x[b:b + 1, :L].clone(), [r], [L])
        nb = int(n_out[b])
        assert y1.shape == (1, nb) and int(n1[0]) == nb
        assert torch.equal(y[b, :nb], y1[0]), (r, L)
        assert not y[b, nb:].any()
    # a device rate outside the set: n_out = 0 and a zero row
    bad = rate_t.clone()
    bad[3] = 12345
    y2, n2 = m(x, bad, len_t)
    assert int(n2[3]) == 0 and not y2[3].any()
    keep = [b for b in range(len(rates)) if b != 3]
    assert torch.equal(y2[keep], y[keep]) and torch.equal(n2[keep], n_out[keep])


def _tone(L, rate, seed):
    t = torch.arange(L, dtype=torch.float64) / rate
    g = torch.Generator().manual_seed(seed)
    x = 0.3 * torch.sin(2 * math.pi * 220 * t) + 0.2 * torch.sin(2 * math.pi * 3100 * t)
    x = x + 0.05 * torch.randn(L, generator=g, dtype=torch.float64)
    return (x * 32767).round().clamp(-32768, 32767).to(torch.int16)


@pytest.fixture(scope="module", params=[24, 48])
def sr(request, hsv):
    which = request.param
    m = (hsv.SpeechSR24 if which == 24 else hsv.SpeechSR48)(100, 40, **hsv.SR_CFG)
    m.load_state_dict(golden_sd(f"speechsr{which}_state.npz"), strict=True)
    return m.to(DEV).eval()


def test_chain_per_item_and_reference(hsv, sr):
    m = hsv.SpeechSRAudio(sr)
    rates = [48000, 44100, 16000, 22050, 8000, 24000, 32000, 11025]
    Ls = [int(r * s) + 3 for r, s in zip(rates, (0.9, 0.55, 0.7, 0.4, 0.8, 0.3, 0.6, 0.5))]
    T = max(Ls) + 100
    x = torch.zeros(len(rates), T, dtype=torch.int16)
    for b, (r, L) in enumerate(zip(rates, Ls)):
        x[b, :L] = _tone(L, r, b)
        x[b, L:] = 12345
    x = x.to(DEV)
    with torch.no_grad():
        out, n_sr = m(x, rates, Ls)
        pcm, n_sr2 = m(x, rates, Ls, pcm16=True)
    assert torch.equal(n_sr, n_sr2) and pcm.dtype == torch.int16
    up, down = m.up, m.down
    for b, (r, L) in enumerate(zip(rates, Ls)):
        nb = int(n_sr[b])
        with torch.no_grad():
            y1, n1 = m.resample(x[b:b + 1, :L].clone(), [r], [L])
            o1 = sr(y1.unsqueeze(1))
        assert nb == int(n1[0]) * up // down == o1.shape[-1]
        assert torch.equal(out[b, 0, :nb], o1[0, 0]) and not out[b, 0, nb:].any()
        assert torch.equal(pcm[b, 0, :nb], hsv.to_pcm16(o1, order="speechsr")[0, 0])
        # the reference chain: torchaudio on the CPU, then the same SpeechSR
        y_ta = _torchaudio_resample(x[b, :L].cpu().float() / 32768.0, r, 16000)
        with torch.no_grad():
            ref = sr(y_ta.view(1, 1, -1).to(DEV))[0, 0].double().cpu().numpy()
        got = out[b, 0, :nb].double().cpu().numpy()
        ma, snr = CF.max_abs(ref, got), CF.snr_db(ref, got)
        assert ma <= MAX_ABS_TOL and snr >= SNR_DB_MIN, (r, ma, snr)


def test_chain_graph_serves_every_mix(hsv, sr):
    m = hsv.SpeechSRAudio(sr)
    runner = hsv.CudaGraphRunner(m)
    B, T, out_len = 4, 48000, 16000
    rng = np.random.default_rng(3)
    for it in range(4):
        rates = [int(r) for r in rng.choice([8000, 16000, 22050, 32000, 44100, 48000], B)]
        Ls = [int(rng.integers(1, min(T, r) + 1)) for r in rates]
        x = torch.randint(-20000, 20000, (B, T), generator=torch.Generator().manual_seed(it),
                          dtype=torch.int32).to(torch.int16).to(DEV)
        rate_t = torch.tensor(rates, dtype=torch.int32, device=DEV)
        len_t = torch.tensor(Ls, dtype=torch.int32, device=DEV)
        with torch.no_grad():
            ref, n_ref = m(x, rate_t, len_t, True, out_len=out_len)
        got, n_got = runner(x, rate_t, len_t, pcm16=True, out_len=out_len)
        assert torch.equal(got, ref) and torch.equal(n_got, n_ref)
    assert runner.captures == 1
