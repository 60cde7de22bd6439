"""SpeechSR from audio at any sample rate: the resampling step of inference_speechsr.py:28-34 on the device.

The reference loads a file at whatever rate it has and resamples it to 16 kHz on the host with
``torchaudio.functional.resample(audio, sr, 16000, resampling_method="kaiser_window")`` before SpeechSR.  ``Resample``
is that operator for a padded batch with one rate and one length per item (``ops.resample``, csrc/resample.cu), and
``SpeechSRAudio`` chains it with the ragged SpeechSR and PCM kernels, all on one stream with nothing read back.  Each
item's result equals, bit for bit, its own batch-1 run.  torchaudio is not needed at run time: the filter tables are
built here with torchaudio's formula and torch ops, in the same order, so they are the same fp32 values.
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch
from torch import nn

from . import ops
from .modules import SpeechSRGenerator, _SpeechSRSynthesizer
from .runtime import ragged_batches

DEFAULT_RATES = (8000, 11025, 16000, 22050, 24000, 32000, 44100, 48000)
# torchaudio's "kaiser_window" (= sinc_interp_kaiser) defaults, the call inference_speechsr.py makes
LOWPASS_FILTER_WIDTH = 6
ROLLOFF = 0.99
BETA = 14.769656459379492
MAX_RATES = 16                 # descriptors the kernel takes
MAX_TABLE_FLOATS = 1 << 24     # one rate pair's filter table (64 MB) at most


def ratio(orig: int, new: int) -> Tuple[int, int, int]:
    """(o, n, width) of resampling orig -> new: o : n = orig : new reduced, width the filter's half-length in input
    samples (torchaudio's ``_get_sinc_resample_kernel``); the filter has K = 2 width + o taps."""
    g = math.gcd(int(orig), int(new))
    o, n = int(orig) // g, int(new) // g
    return o, n, math.ceil(LOWPASS_FILTER_WIDTH * o / (min(o, n) * ROLLOFF))


def sinc_kaiser_table(orig: int, new: int) -> Tuple[torch.Tensor, int]:
    """(fp32 CPU [n, K] filter table, width) of orig -> new: torchaudio's ``_get_sinc_resample_kernel(..., "sinc_interp_
    kaiser", dtype=torch.float32)`` (the dtype of an fp32 waveform), the same torch ops in the same order, so the values
    are identical.  Row p is the filter of output phase p: y[f n + p] = sum_k table[p, k] x[f o + k - width]."""
    o, n, width = ratio(orig, new)
    base_freq = min(o, n) * ROLLOFF
    idx = torch.arange(-width, width + o, dtype=torch.float32)[None, None] / o
    t = torch.arange(0, -n, -1, dtype=torch.float32)[:, None, None] / n + idx
    t *= base_freq
    t = t.clamp_(-LOWPASS_FILTER_WIDTH, LOWPASS_FILTER_WIDTH)
    beta = torch.tensor(float(BETA))
    window = torch.i0(beta * torch.sqrt(1 - (t / LOWPASS_FILTER_WIDTH) ** 2)) / torch.i0(beta)
    t *= math.pi
    scale = base_freq / o
    kernels = torch.where(t == 0, torch.tensor(1.0).to(t), t.sin() / t)
    kernels *= window * scale
    return kernels[:, 0], width


def output_count(L: int, o: int, n: int) -> int:
    """torchaudio's output count for L input samples at o : n: ``ceil(torch.as_tensor(n * L / o))`` -- the fp64
    quotient rounded to fp32, torch's default dtype -- capped at the (L // o + 1) n outputs its conv1d produces.  For
    about 0.4 % of the lengths of 2-15 s at 44.1 kHz it is one below the exact ceil(n L / o)."""
    return min(math.ceil(float(np.float32(n * L / o))), (L // o + 1) * n)


def resampled_lengths(rates: Sequence[int], lengths: Sequence[int], rate_set: Sequence[int] = DEFAULT_RATES,
                      new_freq: int = 16000, T: Optional[int] = None, out_len: Optional[int] = None) -> List[int]:
    """Host mirror of ``Resample``: the ``n_out`` of every item, ``output_count`` (torchaudio's output length), or L
    when the rate is ``new_freq``.  Raises ValueError on a rate outside ``rate_set``, a length
    outside [1, T] (T = None: no upper bound) or an ``out_len`` below some n_out -- requests the device would answer
    with n_out = 0, a clamped length or a cut output."""
    rates, lengths = [int(v) for v in rates], [int(v) for v in lengths]
    if len(rates) != len(lengths):
        raise ValueError(f"{len(rates)} rates for {len(lengths)} lengths")
    known = set(int(r) for r in rate_set)
    out = []
    for b, (r, L) in enumerate(zip(rates, lengths)):
        if r not in known:
            raise ValueError(f"item {b}: rate {r} is not in the resampler's set {sorted(known)}")
        if L < 1 or (T is not None and L > T):
            raise ValueError(f"item {b}: length {L} outside [1, {T if T is not None else 'inf'}]")
        if r == new_freq:
            out.append(L)
        else:
            o, n, _ = ratio(r, new_freq)
            out.append(output_count(L, o, n))
    if out_len is not None and out and max(out) > out_len:
        raise ValueError(f"out_len = {out_len} is below the longest output ({max(out)} samples)")
    return out


def _host_or_device(v, B: int, device, name: str):
    """An int CUDA tensor [B] (never read back) as int32, or a host sequence as a list of ints (checked by the mirror)."""
    if isinstance(v, torch.Tensor):
        if v.device != torch.device(device):
            raise ValueError(f"{name} is on {v.device}, the input is on {device}")
        if tuple(v.shape) != (B,) or v.dtype not in (torch.int32, torch.int64):
            raise ValueError(f"{name} must be an int32 or int64 tensor of shape ({B},)")
        return v.to(torch.int32).contiguous()
    vals = [int(x) for x in v]
    if len(vals) != B:
        raise ValueError(f"{name} has {len(vals)} entries for a batch of {B}")
    return vals


class Resample(nn.Module):
    """``torchaudio.functional.resample(x_b, rate_b, new_freq, resampling_method="kaiser_window")`` of every item of a
    padded batch, on the device (csrc/resample.cu).

    The filter tables of ``rates`` -> ``new_freq`` are built once (``sinc_kaiser_table``) and kept as a non-persistent
    buffer: they follow ``.to()`` and stay out of ``state_dict``.

    ``forward(x, rate, lengths, *, out_len=None) -> (y, n_out)``: x fp32 or int16 PCM (read as s / 32768) CUDA [B, T],
    mono; rate / lengths: int CUDA tensors [B] (never read back, so the call is capturable) or host sequences (checked
    by ``resampled_lengths``).  Item b reads x[b, :lengths[b]] only.  y fp32 [B, out_len]: item b's first n_out[b]
    samples (int32 CUDA [B]) are its resampled audio, the rest is 0; an item whose device rate is not in the set gets
    n_out = 0.  ``out_len`` defaults to the longest output with host rates and lengths, else to ceil(new_freq T /
    min(rates)), which holds every item."""

    def __init__(self, rates: Sequence[int] = DEFAULT_RATES, new_freq: int = 16000):
        super().__init__()
        rates = tuple(int(r) for r in rates)
        if not rates or len(rates) > MAX_RATES or len(set(rates)) != len(rates) or min(rates) < 1 or new_freq < 1:
            raise ValueError(f"rates must be 1 to {MAX_RATES} distinct positive rates, new_freq positive")
        self.rates, self.new_freq = rates, int(new_freq)
        desc, tables, off = [], [], 0
        for r in rates:
            if r == self.new_freq:
                desc.append((r, 1, 1, 0, 0, 0))
                continue
            o, n, width = ratio(r, self.new_freq)
            if (2 * width + o) * n > MAX_TABLE_FLOATS:
                raise ValueError(f"{r} -> {self.new_freq} Hz needs a {2 * width + o} x {n} filter table")
            tab, _ = sinc_kaiser_table(r, self.new_freq)
            desc.append((r, o, n, width, tab.shape[1], off))
            tables.append(tab.t().reshape(-1))     # [K][n]: a warp's consecutive phases read consecutive words
            off += tab.numel()
        self.desc = tuple(desc)
        self.register_buffer("table", torch.cat(tables) if tables else torch.zeros(0), persistent=False)

    def output_lengths(self, rates: Sequence[int], lengths: Sequence[int], T: Optional[int] = None,
                       out_len: Optional[int] = None) -> List[int]:
        """``resampled_lengths`` for this module's rate set and new_freq."""
        return resampled_lengths(rates, lengths, self.rates, self.new_freq, T, out_len)

    def forward(self, x: torch.Tensor, rate, lengths, *, out_len: Optional[int] = None):
        if not isinstance(x, torch.Tensor) or x.dim() != 2:
            raise ValueError("x must be a [B, T] tensor (mono)")
        B, T = x.shape
        rate = _host_or_device(rate, B, x.device, "rate")
        lengths = _host_or_device(lengths, B, x.device, "lengths")
        if isinstance(rate, list) and isinstance(lengths, list):
            n_host = self.output_lengths(rate, lengths, T, out_len)
            if out_len is None:
                out_len = max(n_host + [1])
        else:
            if isinstance(rate, list):
                self.output_lengths(rate, [1] * B)
            elif isinstance(lengths, list):
                if any(not 1 <= v <= T for v in lengths):
                    raise ValueError(f"lengths must lie in [1, {T}]")
            if out_len is None:
                out_len = -(-self.new_freq * T // min(self.rates))
        if int(out_len) < 1:
            raise ValueError("out_len must be >= 1")
        if isinstance(rate, list):
            rate = torch.tensor(rate, dtype=torch.int32, device=x.device)
        if isinstance(lengths, list):
            lengths = torch.tensor(lengths, dtype=torch.int32, device=x.device)
        return ops.resample(x.contiguous(), rate, lengths, self.table, self.desc, self.new_freq, int(out_len))


class SpeechSRAudio(nn.Module):
    """inference_speechsr.py's ``SuperResoltuion`` (:28-41) for a padded batch of audio at any rate of ``rates``:
    ``Resample`` to 16 kHz -> ``sr`` (a loaded ``SpeechSR24`` / ``SpeechSR48``, ragged ``lengths=``) -> optionally the
    per-utterance peak-normalised int16 PCM (``to_pcm16(order="speechsr", per_utterance=True)``).

    ``forward(x, rate, lengths, pcm16=False, *, out_len=None) -> (out [B, 1, out_len * scale], n_sr int32 [B])``: x, rate,
    lengths and out_len (16 kHz samples) as ``Resample.forward``; n_sr = each item's output samples at the SR rate.
    Everything runs on one stream with nothing read back, so one ``CudaGraphRunner`` graph per padded (B, T, out_len)
    serves every mix of rates and lengths.  Item b's output equals, bit for bit, the chain run on that item alone."""

    def __init__(self, sr: nn.Module, rates: Sequence[int] = DEFAULT_RATES):
        super().__init__()
        gen = sr.dec if isinstance(sr, _SpeechSRSynthesizer) else sr
        if not isinstance(gen, SpeechSRGenerator):
            raise TypeError("SpeechSRAudio takes a SpeechSR24 / SpeechSR48 or its generator")
        self.sr = sr
        self.resample = Resample(rates, 16000).to(gen.conv_post.weight.device)
        self.up, self.down = ops.SR_RATIOS[gen.scale]

    def forward(self, x: torch.Tensor, rate, lengths, pcm16: bool = False, *, out_len: Optional[int] = None):
        y, n16 = self.resample(x, rate, lengths, out_len=out_len)
        out = self.sr(y.unsqueeze(1), lengths=n16)
        # int(L * 1.5) == 3 L // 2 and int(L * 3) == 3 L, as SpeechSRGenerator.forward computes them
        n_sr = n16 * self.up // self.down
        if pcm16:
            from .runtime import to_pcm16
            out = to_pcm16(out, order="speechsr", per_utterance=True)
        return out, n_sr


def audio_batches(rates: Sequence[int], lengths: Sequence[int], max_batch: int, rate_set: Sequence[int] = DEFAULT_RATES,
                  new_freq: int = 16000, out_multiple: int = 1600,
                  in_multiple: int = 4800) -> List[Tuple[List[int], int, int]]:
    """Micro-batches of mixed-rate requests for ``SpeechSRAudio`` / ``Resample``: ``runtime.ragged_batches`` of their
    ``new_freq`` lengths (``resampled_lengths``, which rejects bad requests) -> [(ids, T, out_len)], with out_len the
    batch's longest output rounded up to a multiple of ``out_multiple`` and T its longest input rounded up to a multiple
    of ``in_multiple``.  Both roundings bound the number of distinct padded shapes (one captured graph each)."""
    if in_multiple < 1:
        raise ValueError("in_multiple must be >= 1")
    n_out = resampled_lengths(rates, lengths, rate_set, new_freq)
    out = []
    for ids, out_len in ragged_batches(range(len(n_out)), n_out, max_batch, out_multiple):
        longest = max(int(lengths[i]) for i in ids)
        out.append((ids, -(-longest // in_multiple) * in_multiple, out_len))
    return out
