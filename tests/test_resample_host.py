"""Host side of the any-rate SpeechSR input (megatts2_hierspeechpp_b200/resample.py) on the CPU: the filter tables and
output lengths against torchaudio, the host mirror's checks, the fp64 oracle, the batching helper and the C-ABI's
argument errors.  The torchaudio comparisons are skipped where torchaudio is not installed."""
import ctypes
import math
import warnings

import numpy as np
import pytest
import torch

from megatts2_hierspeechpp_b200 import resample as RS

PAIRS = [(r, 16000) for r in RS.DEFAULT_RATES if r != 16000] + [(48000, 44100)]


def _ta():
    ta = pytest.importorskip("torchaudio")
    import torchaudio.functional.functional as taf
    return ta, taf


def _lengths(orig, new):
    o, n, width = RS.ratio(orig, new)
    Ls = {L for L in (1, 2, width - 1, o - 1, o, o + 1, 3 * orig + 17, 10 * orig) if L >= 1}
    # and the first length of 2 s or more whose torchaudio count is below the exact ceil(n L / o), where there is one
    below = [L for L in range(2 * orig, 15 * orig) if RS.output_count(L, o, n) != -(-n * L // o)][:1]
    return sorted(Ls | set(below))


@pytest.mark.parametrize("orig,new", PAIRS)
def test_table_bit_identical_to_torchaudio(orig, new):
    _, taf = _ta()
    g = math.gcd(orig, new)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref, ref_width = taf._get_sinc_resample_kernel(orig, new, g, 6, 0.99, "sinc_interp_kaiser", None,
                                                       torch.device("cpu"), torch.float32)
    tab, width = RS.sinc_kaiser_table(orig, new)
    o, n, w = RS.ratio(orig, new)
    assert width == ref_width == w
    assert tuple(ref.shape) == (n, 1, 2 * width + o)
    assert tab.dtype == torch.float32 and torch.equal(tab, ref[:, 0])


@pytest.mark.parametrize("orig,new", PAIRS)
def test_output_length_matches_torchaudio(orig, new):
    ta, _ = _ta()
    for L in _lengths(orig, new):
        y = ta.functional.resample(torch.zeros(L), orig, new, resampling_method="sinc_interp_kaiser")
        assert RS.resampled_lengths([orig], [L], RS.DEFAULT_RATES + (new,), new) == [y.shape[-1]], L


@pytest.mark.parametrize("orig,new", PAIRS)
def test_output_length_formula_up_to_int32(orig, new):
    # torchaudio's own expression (_apply_sinc_resample_kernel), evaluated without running the resampler
    o, n, _ = RS.ratio(orig, new)
    rng = np.random.default_rng(orig)
    Ls = {2 ** 31 - 1, 2 ** 31 - 2, 2 ** 30, 1, o, o + 1}
    Ls |= {int(v) for v in rng.integers(1, 2 ** 31 - 1, 2000)}
    Ls |= {max(1, int(k) * o + d) for k in rng.integers(1, (2 ** 31 - 2) // o, 200) for d in (-1, 0, 1)}
    for L in sorted(Ls):
        # L a Python int, as torchaudio's waveform.shape gives it: n * L / o is a Python float, as_tensor makes it fp32
        ref = min(int(torch.ceil(torch.as_tensor(n * L / o)).long()), (L // o + 1) * n)   # conv1d gives (L//o+1) n
        assert RS.resampled_lengths([orig], [L], (orig,), new) == [ref], L


def test_identity_rate_length():
    assert RS.resampled_lengths([16000, 48000], [5, 5]) == [5, 2]


def test_mirror_rejects_bad_requests():
    with pytest.raises(ValueError, match="not in"):
        RS.resampled_lengths([44100, 12345], [100, 100])
    with pytest.raises(ValueError, match="outside"):
        RS.resampled_lengths([44100], [0])
    with pytest.raises(ValueError, match="outside"):
        RS.resampled_lengths([44100], [101], T=100)
    with pytest.raises(ValueError, match="out_len"):
        RS.resampled_lengths([48000], [300], out_len=99)
    assert RS.resampled_lengths([48000], [300], out_len=100) == [100]
    with pytest.raises(ValueError, match="rates for"):
        RS.resampled_lengths([48000], [300, 3])


@pytest.mark.parametrize("orig,new", [(44100, 16000), (48000, 16000), (22050, 16000), (8000, 16000),
                                      (48000, 44100)])
def test_fp64_oracle_agrees_with_torchaudio(orig, new):
    from oracle.resample import resample_fp64
    ta, _ = _ta()
    tab, width = RS.sinc_kaiser_table(orig, new)
    o, n, _ = RS.ratio(orig, new)
    x = (torch.rand(3 * orig + 17, generator=torch.Generator().manual_seed(orig)) * 2 - 1)
    y_ta = ta.functional.resample(x, orig, new, resampling_method="sinc_interp_kaiser").numpy().astype(np.float64)
    y64, mag = resample_fp64(x.numpy(), tab.numpy(), o, n, width)
    assert y64.shape == y_ta.shape
    err = np.abs(y_ta - y64)
    K = tab.shape[1]
    assert np.all(err <= K * 2.0 ** -24 * mag)
    # torchaudio's fp32 sums are within a few ulp of the fp64 value for |x| <= 1 (measured: 2.6e-7 absolute)
    assert err.max() <= 1e-6


def test_module_tables_and_descriptors():
    m = RS.Resample()
    assert m.state_dict() == {}
    assert m.table.dtype == torch.float32
    off = 0
    for (rate, o, n, width, K, offset) in m.desc:
        if rate == 16000:
            assert (o, n, width, K) == (1, 1, 0, 0)
            continue
        tab, w = RS.sinc_kaiser_table(rate, 16000)
        assert (o, n, width, K, offset) == (*RS.ratio(rate, 16000)[:2], w, tab.shape[1], off)
        assert torch.equal(m.table[off:off + K * n].view(K, n), tab.t())
        off += K * n
    assert m.table.numel() == off
    with pytest.raises(ValueError):
        RS.Resample(rates=(8000, 8000))
    with pytest.raises(ValueError):
        RS.Resample(rates=tuple(range(8000, 8017)))
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.zeros(1, 100), [44100], [100])


def test_audio_batches_partition_and_bounds():
    rng = np.random.default_rng(7)
    rates = [int(r) for r in rng.choice([16000, 22050, 24000, 32000, 44100, 48000], 97)]
    lengths = [int(rng.integers(2 * r, 15 * r)) for r in rates]
    batches = RS.audio_batches(rates, lengths, 16)
    n16 = RS.resampled_lengths(rates, lengths)
    assert sorted(i for ids, _, _ in batches for i in ids) == list(range(97))
    for ids, T, out_len in batches:
        assert len(ids) <= 16 and T % 4800 == 0 and out_len % 1600 == 0
        assert max(lengths[i] for i in ids) <= T and max(n16[i] for i in ids) <= out_len
    with pytest.raises(ValueError, match="not in"):
        RS.audio_batches([12345], [100], 4)


def test_cabi_argument_errors():
    from megatts2_hierspeechpp_b200 import _lib, build
    build.build()
    lib = _lib.load()
    one = ctypes.c_void_p(16)

    def call(desc, B=1, T=100, T_out=100, table_len=1 << 20, x16=0):
        flat = [v for row in desc for v in row]
        d = (ctypes.c_int32 * max(len(flat), 1))(*flat)
        return lib.hsv_resample_ragged(one, x16, one, one, one, table_len, d, len(desc), 16000, one, one, B, T, T_out,
                                       None)

    good = (48000, 3, 1, 19, 41, 0)
    assert call([good, (16000, 1, 1, 0, 0, 0)], B=0) == 0
    for desc, msg, table_len in (([], b"n_desc", 1 << 20), ([(48000, 3, 1, 19, 40, 0)], b"K == 2 width", 1 << 20),
                                 ([good, good], b"twice", 1 << 20), ([(16000, 1, 1, 1, 3, 0)], b"copy entry", 1 << 20),
                                 ([(48000, 3, 1, 19, 41, 1 << 20)], b"outside", 1 << 20),
                                 ([(44101, 44101, 16000, 17, 44135, 0)], b"window", 1 << 30)):
        rc = call(desc, table_len=table_len)
        assert rc == -1 and msg in lib.hsv_last_error(), (desc, lib.hsv_last_error())
    assert call([good], x16=2) == -1 and b"x_int16" in lib.hsv_last_error()
    assert call([good], T=0) == -1 and b"bad shape" in lib.hsv_last_error()
    rc = lib.hsv_resample_ragged(None, 0, None, None, None, 1 << 20, (ctypes.c_int32 * 6)(*good), 1, 16000, None, None,
                                 1, 100, 100, None)
    assert rc == -1 and b"null table" in lib.hsv_last_error()
    rc = lib.hsv_resample_ragged(None, 0, None, None, one, 1 << 20, (ctypes.c_int32 * 6)(*good), 1, 16000, None, None,
                                 1, 100, 100, None)
    assert rc == -1 and b"null pointer" in lib.hsv_last_error()


def test_graph_runner_keys_keyword_values():
    from megatts2_hierspeechpp_b200.runtime import CudaGraphRunner
    r = CudaGraphRunner(lambda *a, **k: None)
    x = torch.zeros(2, 3)
    assert r._key((x,)) == r._key((x,), {}) == (((2, 3), torch.float32, None),)
    assert r._key((x,), {"out_len": 5}) != r._key((x,), {"out_len": 6})
    assert r._key((x,), {"b": 1, "a": 2}) == r._key((x,), {"a": 2, "b": 1})
    with pytest.raises(TypeError, match="positionally"):
        r._key((x,), {"lengths": x})
