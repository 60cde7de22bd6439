"""Streaming SpeechSR: S concurrent 16 kHz input streams upsampled chunk by chunk in one captured graph, each stream's
concatenated output bit-identical to the offline call on the whole stream.

Each step, every slot's window is the last ``history`` input samples kept on the device plus its new chunk; the windows
form one ragged batch (per-item valid lengths) through the existing ragged SpeechSR kernels, with the interpolation
evaluated at the stream's global indices (``ops.sr_pre_interp_stream``).  Window-edge effects stay inside the halo
(``stream_reach``) and are never emitted; a window that starts at its stream's start or ends at its ``end`` has the
offline call's own edges.  All state lives on the device and is never read back (DESIGN.md §6).
"""
from __future__ import annotations

import math
from typing import List, Sequence, Tuple

import torch
from torch import nn

from . import ops
from .modules import SpeechSRGenerator, _SpeechSRSynthesizer
from .runtime import CudaGraphRunner

# Both ratios need up * L < 2^24: below it fl(L) / fl(L * up / down) == fl(down / up), the scale the stream uses
# (5.8 min of 16 kHz input); past it the offline scale depends on L.
MAX_STREAM_OUTPUT = 1 << 24


def _act_reach(act) -> Tuple[int, int]:
    """(left, right) reach of an ``Activation1d`` in samples of its input: its output t reads x[t - left, t + right],
    the replicate padding of both FIRs included (alias_free_torch/resample.py, filter.py)."""
    up, dn = act.upsample, act.downsample.lowpass
    k_up = up.kernel_size

    def up_range(m):
        # u[m] = y[m + pad_left], y[k] = sum_i xp[i] f[k - ratio * i] (0 <= k - ratio * i < K), xp[i] = x[i - pad]
        lo = -(-(m + up.pad_left - k_up + 1) // up.ratio) - up.pad
        hi = (m + up.pad_left) // up.ratio - up.pad
        return lo, hi

    t = 4 * (k_up + dn.kernel_size)   # any output away from the edges
    # down: out[t] = sum_k f[k] u[stride * t - pad_left + k]
    ms = range(dn.stride * t - dn.pad_left, dn.stride * t - dn.pad_left + dn.kernel_size)
    return t - min(up_range(m)[0] for m in ms), max(up_range(m)[1] for m in ms) - t


def _conv_reach(conv) -> Tuple[int, int]:
    k, d, p = conv.kernel_size[0], conv.dilation[0], conv.padding[0]
    return p, (k - 1) * d - p


def _add(a, b):
    return a[0] + b[0], a[1] + b[1]


def stream_reach(gen: SpeechSRGenerator) -> Tuple[int, int]:
    """(lookahead, left halo) of a streamed SpeechSR generator, in output samples, derived from its layer list.

    Output j of the stream is final once input up to (j + lookahead) / ratio has arrived: the stage (the widest
    resblock: every AMP layer is Activation1d -> conv(k, d) -> Activation1d -> conv(k, 1)), ``activation_post`` and
    ``conv_post`` reach ``post`` output samples to each side; the linear interpolation with ``conv_pre`` (k 7) reads
    input samples floor(src) - 3 ... floor(src) + 1 + 3 of src = (t + 0.5) / ratio - 0.5, plus one sample for the fp32
    rounding of src.  The left halo is the same sum to the other side."""
    nk = gen.num_kernels
    stage = (0, 0)
    for blk in gen.resblocks[:nk]:
        r = (0, 0)
        for i in range(len(blk.dilation)):
            for part in (blk.activations[2 * i], blk.convs1[i], blk.activations[2 * i + 1], blk.convs2[i]):
                r = _add(r, _act_reach(part) if hasattr(part, "upsample") else _conv_reach(part))
        stage = (max(stage[0], r[0]), max(stage[1], r[1]))
    post = _add(_add(stage, _act_reach(gen.activation_post)), _conv_reach(gen.conv_post))
    pl, pr = _conv_reach(gen.conv_pre)
    r = float(gen.scale)
    interp = (math.ceil(r * (pl + 2.5) + 0.5), math.ceil(r * (pr + 2.5) + 0.5))
    return post[1] + interp[1], post[0] + interp[0]


def history_len(lookahead: int, halo: int, ratio: Tuple[int, int]) -> int:
    """Input samples a slot keeps between steps: its next window must start ``halo`` output samples before the first
    output not yet emitted, which lags the input by ``lookahead`` (a multiple of ``down``, so windows start on input
    samples that map to whole output samples)."""
    up, down = ratio
    h = -(-(lookahead + halo) * down // up)
    return -(-h // down) * down


class SRStreamSchedule:
    """Host mirror of a ``SpeechSRStream``'s schedule: from the ``n_new`` / ``start`` / ``end`` the host supplies, the
    ``n_out`` every step returns, without reading anything back.  ``step`` raises ValueError on a request the device
    step would ignore (n_new outside [0, chunk], n_new not a multiple of ``down``, samples or an ``end`` for a slot
    with no open stream) or past the length bound."""

    def __init__(self, slots: int, chunk: int, ratio: Tuple[int, int], lookahead: int):
        self.slots, self.chunk, self.ratio, self.lookahead = slots, chunk, tuple(ratio), lookahead
        self.received = [0] * slots
        self.emitted = [0] * slots
        self.open = [False] * slots

    def step(self, n_new: Sequence[int], start: Sequence, end: Sequence) -> List[int]:
        up, down = self.ratio
        n_new, start, end = [int(v) for v in n_new], [bool(v) for v in start], [bool(v) for v in end]
        if not len(n_new) == len(start) == len(end) == self.slots:
            raise ValueError(f"n_new, start and end need {self.slots} entries each")
        for b, (n, s, e) in enumerate(zip(n_new, start, end)):
            if not 0 <= n <= self.chunk:
                raise ValueError(f"slot {b}: n_new = {n} outside [0, {self.chunk}]")
            if n % down:
                raise ValueError(f"slot {b}: n_new = {n} is odd; a 24 kHz stream takes even chunks (its offline "
                                 "scale is 2/3 only for even lengths)")
            if not (self.open[b] or s) and (n or e):
                raise ValueError(f"slot {b}: {'end' if e else 'samples'} for a slot with no open stream (set start)")
            if ((0 if s else self.received[b]) + n) * up >= MAX_STREAM_OUTPUT:
                raise ValueError(f"slot {b}: the stream reaches 2^24 output samples; its offline scale then "
                                 "depends on its length")
        n_out = []
        for b, (n, s, e) in enumerate(zip(n_new, start, end)):
            if s:
                self.received[b], self.emitted[b], self.open[b] = 0, 0, True
            if not self.open[b]:
                n_out.append(0)
                continue
            self.received[b] += n
            full = self.received[b] * up // down
            done = full if e else max(self.emitted[b], full - self.lookahead)
            n_out.append(done - self.emitted[b])
            self.emitted[b] = done
            if e:
                self.received[b], self.emitted[b], self.open[b] = 0, 0, False
        return n_out


class SpeechSRStream(nn.Module):
    """``slots`` concurrent SpeechSR streams over a loaded ``SpeechSR24`` / ``SpeechSR48`` (or its generator), fed
    ``chunk`` samples at most per slot and step.

    ``step(x_new, n_new, start, end)``: x_new fp32 CUDA [S, chunk]; n_new int32 CUDA [S] the valid new samples per slot
    (0 = idle); start / end bool or int32 CUDA [S]: a new stream begins in the slot (its state is reset) / this is its
    last chunk (an end with n_new = 0 flushes).  Returns (out fp32 [S, capacity], n_out int32 [S]): the samples of each
    slot's stream that became final in this step, out[b, :n_out[b]]; they are the graph's static outputs, valid until
    the next step.  Before its end a stream's output lags its input by ``lookahead`` output samples; at the end
    everything left is flushed.  The concatenation of a stream's outputs equals ``sr(x[None, None])`` bit for bit, for
    any chunking, idle steps and slot reuse.

    24 kHz streams take even n_new only (the offline scale fl(L) / fl(1.5 L) is fl(2/3) for even L alone), and a
    stream must stay below 2^24 output samples (5.8 min of input at 48 kHz).  The device step does not read its inputs
    back: a request that breaks these rules, or sends samples / an end to a slot with no open stream, leaves the slot
    idle.  ``schedule()`` gives a host mirror that checks them and predicts n_out.

    Every step replays one CUDA graph per (slots, chunk); it is captured on an all-idle step (which leaves the state
    unchanged), and again after anything that moves weights or workspaces (``CudaGraphRunner``'s epochs).  Calling the
    module itself runs one step eagerly."""

    def __init__(self, sr: nn.Module, slots: int, chunk: int):
        super().__init__()
        gen = sr.dec if isinstance(sr, _SpeechSRSynthesizer) else sr
        if not isinstance(gen, SpeechSRGenerator):
            raise TypeError("SpeechSRStream takes a SpeechSR24 / SpeechSR48 or its generator")
        if slots < 1 or chunk < 1:
            raise ValueError("slots and chunk must be positive")
        dev = gen.conv_post.weight.device
        if dev.type != "cuda":
            raise RuntimeError(f"SpeechSRStream needs the model on a CUDA device (no CPU fallback), got {dev}")
        self.dec = gen
        self.ratio = ops.SR_RATIOS[gen.scale]
        self.slots, self.chunk = slots, chunk
        self.lookahead, self.halo = stream_reach(gen)
        self.history = history_len(self.lookahead, self.halo, self.ratio)
        up, down = self.ratio
        self.capacity = self.lookahead + -(-chunk * up // down)
        self._hist = torch.zeros(slots, self.history, dtype=torch.float32, device=dev)
        self._state = torch.zeros(slots, 3, dtype=torch.int64, device=dev)
        self._idle = (torch.zeros(slots, chunk, dtype=torch.float32, device=dev),
                      *(torch.zeros(slots, dtype=torch.int32, device=dev) for _ in range(3)))
        self._runner = CudaGraphRunner(self)

    @property
    def captures(self) -> int:
        return self._runner.captures

    def schedule(self) -> SRStreamSchedule:
        """A host mirror of this stream's schedule, starting from all slots closed."""
        return SRStreamSchedule(self.slots, self.chunk, self.ratio, self.lookahead)

    def reset(self):
        """Close every slot."""
        self._hist.zero_()
        self._state.zero_()

    def _args(self, x_new, n_new, start, end):
        dev = self._state.device
        S, N = self.slots, self.chunk
        if not isinstance(x_new, torch.Tensor) or x_new.device != dev or x_new.dtype != torch.float32 \
                or tuple(x_new.shape) != (S, N):
            raise ValueError(f"x_new must be a float32 tensor [{S}, {N}] on {dev}")
        if not isinstance(n_new, torch.Tensor) or n_new.device != dev or n_new.dtype != torch.int32 \
                or tuple(n_new.shape) != (S,):
            raise ValueError(f"n_new must be an int32 tensor [{S}] on {dev}")
        flags = []
        for t, name in ((start, "start"), (end, "end")):
            if not isinstance(t, torch.Tensor) or t.device != dev or t.dtype not in (torch.bool, torch.int32) \
                    or tuple(t.shape) != (S,):
                raise ValueError(f"{name} must be a bool or int32 tensor [{S}] on {dev}")
            flags.append(t.to(torch.int32).contiguous())
        return x_new.contiguous(), n_new.contiguous(), *flags

    def forward(self, x_new, n_new, start, end):
        x_new, n_new, start, end = self._args(x_new, n_new, start, end)
        win, vin, vout, origin, plan = ops.sr_stream_window(x_new, n_new, start, end, self._hist, self._state,
                                                            self.ratio, self.lookahead)
        y = self.dec._stream_forward(win, vin, vout, origin)
        return ops.sr_stream_emit(y.view(self.slots, -1), win, origin, plan, self._hist, self._state, self.capacity)

    def step(self, x_new, n_new, start, end):
        args = self._args(x_new, n_new, start, end)
        if not self._runner.ready(*self._idle):
            # the runner runs the function three times while capturing: do that on an idle step, which changes nothing
            self._runner(*self._idle)
        with torch.no_grad():
            return self._runner(*args)
