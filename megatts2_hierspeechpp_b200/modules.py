"""Drop-in nn.Module mirror of the reference's waveform-generation blocks.

Same class names, constructor signatures, forward signatures and ``state_dict``
keys as the reference (SURVEY.md §8b, Appendix C), so a reference checkpoint
loads ``strict=True`` and the reference's own callers
(``SynthesizerTrn.infer/voice_conversion*`` in hierspeechpp_speechsynthesizer.py
:648-649,670-671,696-697; inference_speechsr.py:38) can use these classes
unchanged.  All arithmetic runs in the sm_100a kernels of ``libhsv.so``:

* ``Activation1d``     -> one fused kernel (alias_free_torch/act.py:23-27)
* AMP block convs      -> tcgen05/TMEM implicit GEMM, fp16 operands, fp32 accumulate,
                          weight-norm folded once per checkpoint (not per forward)
* everything else      -> small fp32 CUDA-core kernels

Inference only (the reference never trains these modules in this repository,
SURVEY.md §2): outputs carry no autograd graph.  CUDA tensors only.
"""
from __future__ import annotations

import math
import warnings
from typing import List, Optional, Sequence

import torch
from torch import nn
from torch.nn import Conv1d, ConvTranspose1d

from . import ops

LRELU_SLOPE = 0.1  # modules.py:17

# 12-tap kaiser-sinc taps (cutoff 0.25, half-width 0.3) as stored in the reference checkpoints
FILTER_TAPS = (0.0020289647, 0.0093894657, -0.0255434588, -0.0576573834, 0.1285725832, 0.4432097971,
               0.4432097971, 0.1285725832, -0.0576573834, -0.0255434588, 0.0093894657, 0.0020289647)


def get_padding(kernel_size: int, dilation: int = 1) -> int:
    """commons.py:14-15."""
    return int((kernel_size * dilation - dilation) / 2)


# Derived tensors (folded / packed weights, the filter check) are cached per module and keyed on the
# parameters' (data_ptr, _version) plus this epoch, which every load_state_dict bumps.  In-place edits
# through ``.data`` bypass autograd's version counter: call ``invalidate_caches()`` after such edits.
_CACHE_EPOCH = [0]


def invalidate_caches():
    _CACHE_EPOCH[0] += 1


def _bump_on_load(module: nn.Module):
    module.register_load_state_dict_post_hook(lambda m, incompatible_keys: invalidate_caches())


def _weight_norm(m: nn.Module) -> nn.Module:
    # old-style weight norm: parameters weight_g / weight_v (the reference's state_dict layout)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return torch.nn.utils.weight_norm(m)


def kaiser_sinc_filter1d(cutoff: float, half_width: float, kernel_size: int) -> torch.Tensor:
    """alias_free_torch/filter.py:28-57 — host-side, constructor only; returns [1,1,k] fp32."""
    even = kernel_size % 2 == 0
    half_size = kernel_size // 2
    delta_f = 4 * half_width
    A = 2.285 * (half_size - 1) * math.pi * delta_f + 7.95
    if A > 50.0:
        beta = 0.1102 * (A - 8.7)
    elif A >= 21.0:
        beta = 0.5842 * (A - 21) ** 0.4 + 0.07886 * (A - 21.0)
    else:
        beta = 0.0
    window = torch.kaiser_window(kernel_size, beta=beta, periodic=False)
    time = (torch.arange(-half_size, half_size) + 0.5) if even else (torch.arange(kernel_size) - half_size)
    if cutoff == 0:
        return torch.zeros(1, 1, kernel_size)
    filt = 2 * cutoff * window * torch.sinc(2 * cutoff * time)
    filt = filt / filt.sum()
    return filt.view(1, 1, kernel_size)


# ----------------------------------------------------------------------------------------------
# alias_free_torch / activations
# ----------------------------------------------------------------------------------------------
class SnakeBeta(nn.Module):
    """activations.py:62-119.  Parameter holder: the arithmetic lives in the fused Activation1d kernel."""

    def __init__(self, in_features, alpha=1.0, alpha_trainable=True, alpha_logscale=False):
        super().__init__()
        self.in_features = in_features
        self.alpha_logscale = alpha_logscale
        if alpha_logscale:
            self.alpha = nn.Parameter(torch.zeros(in_features) * alpha)
            self.beta = nn.Parameter(torch.zeros(in_features) * alpha)
        else:
            self.alpha = nn.Parameter(torch.ones(in_features) * alpha)
            self.beta = nn.Parameter(torch.ones(in_features) * alpha)
        self.alpha.requires_grad = alpha_trainable
        self.beta.requires_grad = alpha_trainable
        self.no_div_by_zero = 0.000000001

    def forward(self, x):
        raise RuntimeError("SnakeBeta is evaluated inside the fused Activation1d kernel on this path; "
                           "wrap it in Activation1d (as every use in the reference does)")


class LowPassFilter1d(nn.Module):
    """alias_free_torch/filter.py:60-94 (buffer holder)."""

    def __init__(self, cutoff=0.5, half_width=0.6, stride: int = 1, padding: bool = True,
                 padding_mode: str = "replicate", kernel_size: int = 12):
        super().__init__()
        if cutoff < -0.0:
            raise ValueError("Minimum cutoff must be larger than zero.")
        if cutoff > 0.5:
            raise ValueError("A cutoff above 0.5 does not make sense.")
        self.kernel_size = kernel_size
        self.even = kernel_size % 2 == 0
        self.pad_left = kernel_size // 2 - int(self.even)
        self.pad_right = kernel_size // 2
        self.stride = stride
        self.padding = padding
        self.padding_mode = padding_mode
        self.register_buffer("filter", kaiser_sinc_filter1d(cutoff, half_width, kernel_size))


class UpSample1d(nn.Module):
    """alias_free_torch/resample.py:10-22 (buffer holder)."""

    def __init__(self, ratio=2, kernel_size=None):
        super().__init__()
        self.ratio = ratio
        self.kernel_size = int(6 * ratio // 2) * 2 if kernel_size is None else kernel_size
        self.stride = ratio
        self.pad = self.kernel_size // ratio - 1
        self.pad_left = self.pad * self.stride + (self.kernel_size - self.stride) // 2
        self.pad_right = self.pad * self.stride + (self.kernel_size - self.stride + 1) // 2
        self.register_buffer("filter", kaiser_sinc_filter1d(0.5 / ratio, 0.6 / ratio, self.kernel_size))


class DownSample1d(nn.Module):
    """alias_free_torch/resample.py:36-44 (buffer holder)."""

    def __init__(self, ratio=2, kernel_size=None):
        super().__init__()
        self.ratio = ratio
        self.kernel_size = int(6 * ratio // 2) * 2 if kernel_size is None else kernel_size
        self.lowpass = LowPassFilter1d(cutoff=0.5 / ratio, half_width=0.6 / ratio, stride=ratio,
                                       kernel_size=self.kernel_size)


class Activation1d(nn.Module):
    """alias_free_torch/act.py:8-27: x2 kaiser-sinc upsample -> SnakeBeta -> x2 low-pass downsample,
    as ONE fused kernel (``hsv_act1d_snakebeta``)."""

    def __init__(self, activation, up_ratio: int = 2, down_ratio: int = 2, up_kernel_size: int = 12,
                 down_kernel_size: int = 12):
        super().__init__()
        if (up_ratio, down_ratio, up_kernel_size, down_kernel_size) != (2, 2, 12, 12):
            raise NotImplementedError("the fused kernel implements the configuration the reference uses: "
                                      "ratio 2/2, 12-tap filters")
        if not isinstance(activation, SnakeBeta) or not activation.alpha_logscale:
            raise NotImplementedError("the fused kernel implements SnakeBeta(alpha_logscale=True), the only "
                                      "activation on the reference's waveform path")
        self.up_ratio = up_ratio
        self.down_ratio = down_ratio
        self.act = activation
        self.upsample = UpSample1d(up_ratio, up_kernel_size)
        self.downsample = DownSample1d(down_ratio, down_kernel_size)
        self._filter_key = None
        _bump_on_load(self)

    def check_filters(self):
        """The kernel constant-folds the taps; the state_dict buffers must equal them (SURVEY.md §0.7)."""
        fu, fd = self.upsample.filter, self.downsample.lowpass.filter
        key = (fu._version, fd._version, fu.data_ptr(), fd.data_ptr(), _CACHE_EPOCH[0])
        if key == self._filter_key:
            return
        ref = torch.tensor(FILTER_TAPS, dtype=torch.float32)
        for name, f in (("upsample.filter", fu), ("downsample.lowpass.filter", fd)):
            if f.numel() != 12 or (f.detach().flatten().cpu().float() - ref).abs().max().item() > 1e-7:
                raise ValueError(f"{name} differs from kaiser_sinc_filter1d(0.25, 0.3, 12); the fused kernel "
                                 "constant-folds those taps")
        self._filter_key = key

    def params(self):
        return self.act.alpha.detach(), self.act.beta.detach()

    def forward(self, x):
        self.check_filters()
        x = _as_input(x)
        a, b = self.params()
        return ops.act1d(x, a, b)


def _as_input(x: torch.Tensor) -> torch.Tensor:
    if not x.is_cuda:
        raise RuntimeError(f"expected a CUDA tensor (no CPU fallback), got device {x.device}")
    if x.dtype != torch.float32:
        raise ValueError(f"expected float32 input, got {x.dtype}")
    return x.detach().contiguous()


# ----------------------------------------------------------------------------------------------
# folded-weight cache (weight norm is folded once per checkpoint instead of every forward)
# ----------------------------------------------------------------------------------------------
class _Folded:
    """Derived tensors of one conv: folded fp32 weight and, on demand, the packed tcgen05 operand."""

    def __init__(self, conv: nn.Module):
        self.conv = conv
        self.key = None
        self.w = None
        self.packed = None
        self.n_tile = None

    def _params(self):
        c = self.conv
        if hasattr(c, "weight_g"):
            return (c.weight_g, c.weight_v)
        return (c.weight,)

    def weight(self) -> torch.Tensor:
        ps = self._params()
        key = tuple((p.data_ptr(), p._version) for p in ps) + (_CACHE_EPOCH[0],)
        if key != self.key:
            if len(ps) == 2:
                g, v = ps
                self.w = ops.weight_norm_fold(v.detach().contiguous(), g.detach().contiguous())
            else:
                self.w = ps[0].detach().contiguous()
            self.packed = None
            self.key = key
        return self.w

    def packed_weight(self, row_tiles: int = 1 << 30, n_tile: Optional[int] = None):
        """(packed fp16 operand stream, n_tile) for a launch with ``row_tiles`` 128-row tiles (x batch), or for
        the given ``n_tile``."""
        w = self.weight()
        if self.packed is None:
            self.packed = {}
        nt = n_tile if n_tile is not None else ops.pick_n_tile(w.shape[0], row_tiles, w.shape[1] * w.shape[2])
        if nt not in self.packed:
            self.packed[nt] = ops.pack_conv_weight(w, nt)
        return self.packed[nt], nt

    def packedT_weight(self, u: int, row_tiles: int = 1 << 30):
        w = self.weight()
        if self.packed is None:
            self.packed = {}
        nt = ops.pick_n_tile(w.shape[1], row_tiles * u)
        if nt not in self.packed:
            self.packed[nt] = ops.pack_convT_weight(w, u, nt)
        return self.packed[nt], nt

    def bias(self):
        b = getattr(self.conv, "bias", None)
        return None if b is None else b.detach()


def _row_tiles(B: int, L: int) -> int:
    return B * ((L + ops.TILE_M - 1) // ops.TILE_M)


# Whole-layer fusion (SURVEY.md §8f1): AMP half-layers whose channel count is at most this run as ONE kernel
# (activation evaluated inside the conv CTA, bit-identical results).  Measured on B200 (DESIGN.md §4) it is
# SLOWER than the act kernel + conv kernel pair -- the activation is FP32-issue-bound and needs ~24 resident
# warps per SM, the fused CTA (144 registers, 66 KB) allows 12 -- so the default is 0 (off); set
# HSV_FUSE_MAX_C=32|64 or FUSE_MAX_CHANNELS[0] to use it.
FUSE_MAX_CHANNELS = [int(__import__("os").environ.get("HSV_FUSE_MAX_C", "0"))]
# ... and only for layers of at most this many elements (B*C*L): small layers are latency-bound (one wave or less per
# kernel), there the saved launch on the critical path is worth more than the slower in-CTA activation
FUSE_MAX_ELEMS = [int(__import__("os").environ.get("HSV_FUSE_MAX_ELEMS", str(1 << 62)))]

# ----------------------------------------------------------------------------------------------
# ragged batches: utterances of different lengths padded to one T
# ----------------------------------------------------------------------------------------------
def _lengths_tensor(lengths, B: int, T: int, device) -> Optional[torch.Tensor]:
    """``lengths`` (per utterance, in the module's input time units) as a contiguous int32 [B] tensor on ``device``.
    A CUDA tensor is only checked for shape / device / dtype -- never read back, so the call stays free of host syncs and
    capturable (the kernels clamp its values to the tensor length); a host sequence is range-checked (1 <= len <= T)."""
    if lengths is None:
        return None
    device = torch.device(device)
    if isinstance(lengths, torch.Tensor):
        if lengths.device != device:
            raise ValueError(f"lengths is on {lengths.device}, the input is on {device}")
        if tuple(lengths.shape) != (B,):
            raise ValueError(f"lengths must have shape ({B},), got {tuple(lengths.shape)}")
        if lengths.dtype not in (torch.int32, torch.int64):
            raise ValueError(f"lengths must be int32 or int64, got {lengths.dtype}")
        return lengths.to(torch.int32).contiguous()
    vals = [int(v) for v in lengths]
    if len(vals) != B:
        raise ValueError(f"lengths has {len(vals)} entries for a batch of {B}")
    bad = [v for v in vals if not 1 <= v <= T]
    if bad:
        raise ValueError(f"lengths must lie in [1, {T}], got {bad[:4]}")
    return torch.tensor(vals, dtype=torch.int32, device=device)


def _length_table(lengths, B: int, T: int, device, mults: Sequence[int]) -> Optional[torch.Tensor]:
    """int32 [len(mults), B] on the device: row i = the valid lengths at the stage whose length is mults[i] x the input's
    (computed once per forward; its rows are the ``valid_len`` of that stage's kernels)."""
    ln = _lengths_tensor(lengths, B, T, device)
    return None if ln is None else torch.stack([ln * m for m in mults])


def _scale_lengths(lengths, m: int):
    """``lengths`` in units m times finer (a device tensor stays on the device)."""
    if lengths is None or isinstance(lengths, torch.Tensor):
        return None if lengths is None else lengths * m
    return [int(v) * m for v in lengths]


def _frame_mask(vl: torch.Tensor, L: int) -> torch.Tensor:
    """fp32 [B, L] 0/1 mask of the valid steps (the operand-writing conv epilogues multiply by it: v * 1.0f is exact)."""
    return (torch.arange(L, device=vl.device, dtype=torch.int32).unsqueeze(0) < vl.unsqueeze(1)).float()


def _vl(valid_len: Optional[torch.Tensor]) -> dict:
    # the ops keep their unragged call when there are no lengths
    return {} if valid_len is None else {"valid_len": valid_len}


def _hops(rates: Sequence[int]) -> List[int]:
    """Length of the input and of every up-sampling stage's output, in input steps."""
    out = [1]
    for u in rates:
        out.append(out[-1] * u)
    return out


_MAIN_SLOT = 3   # blk16 workspace slot of the main stream (slots 0..2 belong to the per-resblock streams)
_DB_SLOT = 15   # second operand workspace of the DBlock's conv chain
_PRE_SLOT = 7    # ... of Generator.pre when Vocoder runs it beside the SourceNetwork (4..6: front.py, 8+: tests)


def _dense_conv(x: torch.Tensor, f: _Folded, k: int, d: int = 1, lrelu: bool = False,
                residual: Optional[torch.Tensor] = None, slot: Optional[int] = None,
                out: Optional[torch.Tensor] = None, valid_len: Optional[torch.Tensor] = None) -> torch.Tensor:
    """'same' Conv1d of an fp32 [B,C,L] tensor: tcgen05 path when both channel counts are multiples of
    16 (pack to the fp16 operand layout, optional leaky_relu(0.1) fused into the pack), fp32 direct
    kernel otherwise.  ``valid_len`` (int32 [B]): the operand is zero past each item's length, so the output below it
    equals the item's own run (the output past it is not meaningful)."""
    B, C, L = x.shape
    cout = f.conv.out_channels
    if C % 16 == 0 and cout % 16 == 0 and ((k - 1) // 2) * d <= ops.BLK_PAD:
        buf = ops.blk16_buffer(B, C, L, x.device, _MAIN_SLOT if slot is None else slot)
        ops.pack_blk16(x, buf, lrelu, **_vl(valid_len))
        ops.check_saturation(buf, C, L)
        wp, nt = f.packed_weight(_row_tiles(B, L))
        return ops.conv1d_umma(buf, wp, f.bias(), L, C, cout, k, d, nt, residual=residual, out=out)
    if valid_len is not None:
        raise NotImplementedError("per-utterance lengths need channel counts that are multiples of 16 here")
    pad = ((k - 1) // 2) * d
    if residual is not None:
        if out is None:
            out = residual.clone()
        else:
            out.copy_(residual)
        return ops.conv1d_direct(x, f.weight(), f.bias(), d=d, pad=pad,
                                 flags=(ops.CONV_LRELU_IN if lrelu else 0) | ops.CONV_ADD_OUT, out=out)
    return ops.conv1d_direct(x, f.weight(), f.bias(), d=d, pad=pad, flags=ops.CONV_LRELU_IN if lrelu else 0, out=out)


def _dense_convT(x: torch.Tensor, f: _Folded, k: int, u: int, add: Optional[torch.Tensor] = None,
                 scale: float = 1.0, valid_len: Optional[torch.Tensor] = None) -> torch.Tensor:
    """ConvTranspose1d(k, stride u, padding (k-u)//2) of the fp32 [B,C,L] tensor ``x * scale`` (+ optional add).
    ``x`` may be the list of per-resblock outputs of the previous stage (``sum_of_blocks(..., separate=True)``): their
    sum is taken inside the operand pack.  ``valid_len`` (int32 [B], input steps): the operand is zero past each item's
    length, so the output below u * length equals the item's own run."""
    B, C, L = (x[0] if isinstance(x, (list, tuple)) else x).shape
    cout = f.conv.out_channels
    if C % 16 == 0 and cout % 16 == 0:
        buf = ops.blk16_buffer(B, C, L, f.weight().device, _MAIN_SLOT)
        ops.pack_blk16(x, buf, scale=scale, **_vl(valid_len))
        ops.check_saturation(buf, C, L)
        wp, nt = f.packedT_weight(u, _row_tiles(B, L))
        return ops.conv_transpose1d_umma(buf, wp, f.bias(), L, C, cout, k, u, nt, add=add)
    if valid_len is not None:
        raise NotImplementedError("per-utterance lengths need channel counts that are multiples of 16 here")
    if scale != 1.0 or isinstance(x, (list, tuple)):
        raise NotImplementedError("channel counts that are not multiples of 16 are not supported on this path")
    return ops.conv_transpose1d(x, f.weight(), f.bias(), u, add=add)


# ----------------------------------------------------------------------------------------------
# AMP block
# ----------------------------------------------------------------------------------------------
class AMPBlock1(nn.Module):
    """hierspeechpp_speechsynthesizer.py:344-392 (AMPBlock0 of speechsr.py:16-64 is identical)."""

    def __init__(self, channels, kernel_size=3, dilation=(1, 3, 5), activation=None):
        super().__init__()
        self.channels = channels
        self.kernel_size = kernel_size
        self.dilation = tuple(dilation)
        self.convs1 = nn.ModuleList([
            _weight_norm(Conv1d(channels, channels, kernel_size, 1, dilation=d, padding=get_padding(kernel_size, d)))
            for d in self.dilation])
        self.convs2 = nn.ModuleList([
            _weight_norm(Conv1d(channels, channels, kernel_size, 1, dilation=1, padding=get_padding(kernel_size, 1)))
            for _ in self.dilation])
        self.num_layers = len(self.convs1) + len(self.convs2)
        self.activations = nn.ModuleList([
            Activation1d(activation=SnakeBeta(channels, alpha_logscale=True)) for _ in range(self.num_layers)])
        self._f1 = [_Folded(c) for c in self.convs1]
        self._f2 = [_Folded(c) for c in self.convs2]
        _bump_on_load(self)

    def run(self, x: torch.Tensor, slot: int = 0, acc: Optional[torch.Tensor] = None, acc_mode: int = ops.ACC_NONE,
            before_final=None, valid_len: Optional[torch.Tensor] = None) -> Optional[torch.Tensor]:
        """x fp32 [B,C,L] (not modified).  Returns the block output, or None when the result is only
        accumulated into ``acc`` (sum over resblocks).  ``before_final`` is called right before the
        last conv is enqueued (used to order accumulation across streams).  ``valid_len`` (int32 [B]): item b is
        x[b, :, :valid_len[b]]; the output below that equals the item's own run, past it it is not meaningful."""
        B, C, L = x.shape
        if C != self.channels or C % 16:
            raise ValueError(f"AMP block expects {self.channels} channels (multiple of 16), got {C}")
        k = self.kernel_size
        fused = C in ops.FUSED_CIN and C <= FUSE_MAX_CHANNELS[0] and B * C * L <= FUSE_MAX_ELEMS[0]
        if fused and valid_len is not None:
            raise NotImplementedError("the fused act+conv half-layer (HSV_FUSE_MAX_C) takes no per-utterance lengths")
        buf = None if fused else ops.blk16_buffer(B, C, L, x.device, slot)
        xt = torch.empty_like(x)
        cur = x
        nl = len(self.dilation)
        for i, d in enumerate(self.dilation):
            a1, a2 = self.activations[2 * i], self.activations[2 * i + 1]
            a1.check_filters(); a2.check_filters()
            last = i == nl - 1
            if fused:
                # act -> conv as one kernel per half-layer (the fp16 operand stays in shared memory)
                w1, _ = self._f1[i].packed_weight(n_tile=C)
                w2, _ = self._f2[i].packed_weight(n_tile=C)
                ops.act_conv1d_umma(cur, *a1.params(), w1, self._f1[i].bias(), C, k, d, out=xt)
                if last and before_final is not None:
                    before_final()
                if last and acc_mode != ops.ACC_NONE:
                    ops.act_conv1d_umma(xt, *a2.params(), w2, self._f2[i].bias(), C, k, 1, residual=cur, acc=acc,
                                        acc_mode=acc_mode, want_out=False)
                    return None
                out = torch.empty_like(x) if cur is x else cur
                ops.act_conv1d_umma(xt, *a2.params(), w2, self._f2[i].bias(), C, k, 1, residual=cur, out=out)
                cur = out
                continue
            w1, nt1 = self._f1[i].packed_weight(_row_tiles(B, L))
            w2, nt2 = self._f2[i].packed_weight(_row_tiles(B, L))
            ops.act1d_blk16(cur, *a1.params(), buf, **_vl(valid_len))
            ops.check_saturation(buf, C, L)
            ops.conv1d_umma(buf, w1, self._f1[i].bias(), L, C, C, k, d, nt1, out=xt)
            ops.act1d_blk16(xt, *a2.params(), buf, **_vl(valid_len))
            ops.check_saturation(buf, C, L)
            if last and before_final is not None:
                before_final()
            if last and acc_mode != ops.ACC_NONE:
                ops.conv1d_umma(buf, w2, self._f2[i].bias(), L, C, C, k, 1, nt2, residual=cur, acc=acc,
                                acc_mode=acc_mode, want_out=False)
                return None
            out = torch.empty_like(x) if cur is x else cur
            ops.conv1d_umma(buf, w2, self._f2[i].bias(), L, C, C, k, 1, nt2, residual=cur, out=out)
            cur = out
        return cur

    def forward(self, x):
        return self.run(_as_input(x))

    def remove_weight_norm(self):
        for l in list(self.convs1) + list(self.convs2):
            torch.nn.utils.remove_weight_norm(l)
        self._f1 = [_Folded(c) for c in self.convs1]
        self._f2 = [_Folded(c) for c in self.convs2]


AMPBlock0 = AMPBlock1


_PRE_OVERLAP = [__import__("os").environ.get("HSV_PRE_OVERLAP", "1") != "0"]      # A/B switch of the pre-stage side streams
# ... which pay while the kernels are short (batch 1: -4.7 % on the step); at batch 16 (40 M elements per late-stage tensor) the
# chained epilogues are 0.5 % faster (A/B on one box), hence the size cut
SEPARATE_MAX_ELEMS = [1 << 23]
_SEPARATE = [__import__("os").environ.get("HSV_SEPARATE_SUMS", "1") != "0"]   # A/B switch of the consumer-side resblock sums


def sum_of_blocks(x: torch.Tensor, blocks: Sequence[AMPBlock1], parallel: bool = False, separate: bool = False,
                  valid_len: Optional[torch.Tensor] = None):
    """(xs, scale) with xs = sum_j resblock_j(x) and scale = 1/num_kernels
    (hierspeechpp_speechsynthesizer.py:440-446).  The sum is accumulated in the epilogue of each block's
    last conv (store, then red.add in stream order: deterministic); the division is applied by the
    consumer of xs (``in_scale`` of the next activation / operand pack), so xs is never re-read.

    ``separate=True`` (multi-stream mode only, up to three blocks): every block writes its own tensor and the LIST is
    returned; the consumer's operand pack adds them in the same fixed order ((x1 + x2) + x3, bit-identical to the
    chained accumulation, same bytes moved).  The last convs of the blocks then run concurrently instead of one
    after the other: at batch 1 that chain was ~10 us at the end of every stage.

    ``valid_len`` (int32 [B]) is passed to every block (``AMPBlock1.run``)."""
    nk = len(blocks)
    if nk == 1:
        return blocks[0].run(x, **_vl(valid_len)), 1.0
    if separate and parallel and nk <= 3 and _SEPARATE[0] and x.numel() <= SEPARATE_MAX_ELEMS[0]:
        main = torch.cuda.current_stream()
        fork = torch.cuda.Event()
        fork.record(main)
        streams = _side_streams(x.device, nk)
        outs = []
        for j, blk in enumerate(blocks):
            s = streams[j]
            s.wait_event(fork)
            with torch.cuda.stream(s):
                outs.append(blk.run(x, slot=j, **_vl(valid_len)))
                ev = torch.cuda.Event()
                ev.record(s)
            main.wait_event(ev)
        return outs, 1.0 / nk
    xs = torch.empty_like(x)
    modes = [ops.ACC_SET] + [ops.ACC_ADD] * (nk - 1)
    if not parallel:
        for j, blk in enumerate(blocks):
            blk.run(x, slot=0, acc=xs, acc_mode=modes[j], **_vl(valid_len))
        return xs, 1.0 / nk
    # one stream per resblock; the accumulating epilogues are chained with events
    main = torch.cuda.current_stream()
    fork = torch.cuda.Event()
    fork.record(main)
    streams = _side_streams(x.device, nk)
    done = [torch.cuda.Event() for _ in range(nk)]
    for j, blk in enumerate(blocks):
        s = streams[j]
        s.wait_event(fork)
        with torch.cuda.stream(s):
            prev = done[j - 1] if j > 0 else None
            blk.run(x, slot=j, acc=xs, acc_mode=modes[j],
                    before_final=(lambda p=prev, st=s: st.wait_event(p)) if prev is not None else None,
                    **_vl(valid_len))
            done[j].record(s)
    for ev in done:
        main.wait_event(ev)
    return xs, 1.0 / nk


_streams = {}


def _side_streams(device, n):
    key = (torch.device(device).index, n)
    if key not in _streams:
        _streams[key] = [torch.cuda.Stream(device=device) for _ in range(n)]
    return _streams[key]


# ----------------------------------------------------------------------------------------------
# HierSpeech++ vocoder blocks
# ----------------------------------------------------------------------------------------------
class DBlock(nn.Module):
    """hierspeechpp_speechsynthesizer.py:317-342."""

    def __init__(self, input_size, hidden_size, factor):
        super().__init__()
        self.factor = factor
        self.residual_dense = _weight_norm(Conv1d(input_size, hidden_size, 1))
        self.conv = nn.ModuleList([
            _weight_norm(Conv1d(input_size, hidden_size, 3, dilation=1, padding=1)),
            _weight_norm(Conv1d(hidden_size, hidden_size, 3, dilation=2, padding=2)),
            _weight_norm(Conv1d(hidden_size, hidden_size, 3, dilation=4, padding=4)),
        ])
        self._fr = _Folded(self.residual_dense)
        self._fc = [_Folded(c) for c in self.conv]
        _bump_on_load(self)

    def forward(self, x, side=None, *, valid_len: Optional[torch.Tensor] = None):
        """``side`` = (stream, workspace slot): run the residual 1x1 conv there, beside the first two convs of the
        main branch (it is only needed by the third).  ``valid_len`` (int32 [B], OUTPUT steps, i.e. input steps /
        factor): the output below it equals each item's own run."""
        x = _as_input(x)
        size = x.shape[-1] // self.factor
        # nearest down-sampling commutes with the 1x1 conv: gather first (4x less work, same values)
        xd = ops.nearest_gather(x, size)
        mask = None if valid_len is None else _frame_mask(valid_len, size)
        if side is None:
            res = _dense_conv(xd, self._fr, 1, valid_len=valid_len)
            ready = None
        else:
            st, slot = side
            main = torch.cuda.current_stream()
            res = torch.empty(x.shape[0], self.residual_dense.out_channels, size, dtype=torch.float32, device=x.device)
            fork, ready = torch.cuda.Event(), torch.cuda.Event()
            fork.record(main)
            st.wait_event(fork)
            with torch.cuda.stream(st):
                _dense_conv(xd, self._fr, 1, slot=slot, out=res, valid_len=valid_len)
                ready.record(st)
        B, cin, L = xd.shape
        hid = self.conv[0].out_channels
        if cin % 16 == 0 and hid % 16 == 0:
            # leaky_relu -> conv chain with operand-writing epilogues: one pack, then every conv hands the next one its
            # fp16 operand (leaky_relu applied in the epilogue)
            rt = _row_tiles(B, L)
            b0 = ops.blk16_buffer(B, cin, L, xd.device, _MAIN_SLOT)
            ops.pack_blk16(xd, b0, True, **_vl(valid_len))
            ops.check_saturation(b0, cin, L)
            b1 = ops.blk16_buffer(B, hid, L, xd.device, _MAIN_SLOT)
            b2 = ops.blk16_buffer(B, hid, L, xd.device, _DB_SLOT)
            # with lengths, the mask gives each operand the zero tail of the item's own run
            w0, n0 = self._fc[0].packed_weight(rt)
            ops.conv1d_umma_blk(b0, w0, self._fc[0].bias(), L, cin, hid, 3, 1, n0, b1, ops.BLK_LRELU, mask=mask)
            w1, n1 = self._fc[1].packed_weight(rt)
            ops.conv1d_umma_blk(b1, w1, self._fc[1].bias(), L, hid, hid, 3, 2, n1, b2, ops.BLK_LRELU, mask=mask)
            ops.check_saturation(b2, hid, L)
            if ready is not None:
                torch.cuda.current_stream().wait_event(ready)
            w2, n2 = self._fc[2].packed_weight(rt)
            return ops.conv1d_umma(b2, w2, self._fc[2].bias(), L, hid, hid, 3, 4, n2, residual=res)
        h = xd
        for i, d in enumerate((1, 2, 4)):
            if i == 2 and ready is not None:
                torch.cuda.current_stream().wait_event(ready)
            h = _dense_conv(h, self._fc[i], 3, d, lrelu=True, residual=res if i == 2 else None, valid_len=valid_len)
        return h

    def remove_weight_norm(self):
        for l in self.conv:
            torch.nn.utils.remove_weight_norm(l)
        self._fc = [_Folded(c) for c in self.conv]


class _VocoderBase(nn.Module):
    parallel_blocks = False

    def __init__(self):
        super().__init__()
        _bump_on_load(self)

    def _stage(self, x, i, separate: bool = False, valid_len: Optional[torch.Tensor] = None):
        """``separate``: the consumer of this stage is an operand pack (the next stage's ConvTranspose1d), which can
        take the per-resblock tensors as a list."""
        nk = self.num_kernels
        return sum_of_blocks(x, [self.resblocks[i * nk + j] for j in range(nk)], self.parallel_blocks, separate,
                             valid_len)

    def _length_table(self, lengths, x: torch.Tensor) -> Optional[torch.Tensor]:
        """Valid lengths of the input and of every up-sampling stage's output (rows of an int32 [stages + 1, B])."""
        return _length_table(lengths, x.shape[0], x.shape[-1], x.device, _hops(self.upsample_rates))


class SourceNetwork(_VocoderBase):
    """hierspeechpp_speechsynthesizer.py:251-308."""

    def __init__(self, upsample_initial_channel=256):
        super().__init__()
        resblock_kernel_sizes = [3, 5, 7]
        upsample_rates = [2, 2]
        initial_channel = 192
        upsample_kernel_sizes = [4, 4]
        resblock_dilation_sizes = [[1, 3, 5], [1, 3, 5], [1, 3, 5]]
        self.num_kernels = len(resblock_kernel_sizes)
        self.num_upsamples = len(upsample_rates)
        self.upsample_rates = upsample_rates
        self.conv_pre = _weight_norm(Conv1d(initial_channel, upsample_initial_channel, 7, 1, padding=3))
        self.ups = nn.ModuleList()
        for i, (u, k) in enumerate(zip(upsample_rates, upsample_kernel_sizes)):
            self.ups.append(_weight_norm(ConvTranspose1d(upsample_initial_channel // (2 ** i),
                                                         upsample_initial_channel // (2 ** (i + 1)), k, u,
                                                         padding=(k - u) // 2)))
        self.resblocks = nn.ModuleList()
        ch = upsample_initial_channel
        for i in range(len(self.ups)):
            ch = upsample_initial_channel // (2 ** (i + 1))
            for k, d in zip(resblock_kernel_sizes, resblock_dilation_sizes):
                self.resblocks.append(AMPBlock1(ch, k, d, activation="snakebeta"))
        self.activation_post = Activation1d(activation=SnakeBeta(ch, alpha_logscale=True))
        self.conv_post = Conv1d(ch, 1, 7, 1, padding=3, bias=False)
        self.cond = Conv1d(256, upsample_initial_channel, 1)
        self._f_pre = _Folded(self.conv_pre)
        self._f_ups = [_Folded(u) for u in self.ups]
        self._f_post = _Folded(self.conv_post)
        self._f_cond = _Folded(self.cond)

    def forward(self, x, g, need_pred: bool = True, *, lengths=None):
        """Returns (e, e_) like the reference (:290-308).  ``need_pred=False`` skips the f0 predictor
        ``conv_post`` (e_ is returned as None): ``Generator`` only consumes the hidden state e.

        ``lengths`` (frames of x per utterance: int CUDA tensor [B] or host sequence): a padded batch of utterances of
        different lengths; item b's outputs below 4 * lengths[b] equal its own unpadded run, the rest is 0."""
        x, g = _as_input(x), _as_input(g)
        V = self._length_table(lengths, x)
        vl = (lambda i: None) if V is None else (lambda i: V[i])
        xp = _dense_conv(x, self._f_pre, 7, valid_len=vl(0))
        cg = ops.conv1d_direct(g, self._f_cond.weight(), self._f_cond.bias())
        x = ops.add3_bcast(xp, None, cg, out=xp)
        sc = 1.0
        for i in range(self.num_upsamples):
            x = _dense_convT(x, self._f_ups[i], self.ups[i].kernel_size[0], self.upsample_rates[i], scale=sc,
                             valid_len=vl(i))
            x, sc = self._stage(x, i, separate=i < self.num_upsamples - 1, valid_len=vl(i + 1))
        self.activation_post.check_filters()
        n = self.num_upsamples
        x = ops.act1d(x, *self.activation_post.params(), scale=sc, **_vl(vl(n)))
        x_ = ops.conv1d_direct(x, self._f_post.weight(), None, pad=3, **_vl(vl(n))) if need_pred else None
        return x, x_


class Generator(_VocoderBase):
    """HierSpeech++ BigVGAN-style generator, hierspeechpp_speechsynthesizer.py:394-461."""

    def __init__(self, initial_channel, resblock_kernel_sizes, resblock_dilation_sizes, upsample_rates,
                 upsample_initial_channel, upsample_kernel_sizes, gin_channels=256):
        super().__init__()
        self.num_kernels = len(resblock_kernel_sizes)
        self.num_upsamples = len(upsample_rates)
        self.upsample_rates = list(upsample_rates)
        self.conv_pre = _weight_norm(Conv1d(initial_channel, upsample_initial_channel, 7, 1, padding=3))
        self.ups = nn.ModuleList()
        for i, (u, k) in enumerate(zip(upsample_rates, upsample_kernel_sizes)):
            self.ups.append(_weight_norm(ConvTranspose1d(upsample_initial_channel // (2 ** i),
                                                         upsample_initial_channel // (2 ** (i + 1)), k, u,
                                                         padding=(k - u) // 2)))
        self.resblocks = nn.ModuleList()
        ch = upsample_initial_channel
        for i in range(len(self.ups)):
            ch = upsample_initial_channel // (2 ** (i + 1))
            for k, d in zip(resblock_kernel_sizes, resblock_dilation_sizes):
                self.resblocks.append(AMPBlock1(ch, k, d, activation="snakebeta"))
        self.activation_post = Activation1d(activation=SnakeBeta(ch, alpha_logscale=True))
        self.conv_post = Conv1d(ch, 1, 7, 1, padding=3, bias=False)
        if gin_channels != 0:
            self.cond = nn.Conv1d(gin_channels, upsample_initial_channel, 1)
        self.downs = DBlock(upsample_initial_channel // 8, upsample_initial_channel, 4)
        self.proj = Conv1d(upsample_initial_channel // 8, upsample_initial_channel // 2, 7, 1, padding=3)
        self._f_pre = _Folded(self.conv_pre)
        self._f_ups = [_Folded(u) for u in self.ups]
        self._f_post = _Folded(self.conv_post)
        self._f_cond = _Folded(self.cond) if gin_channels != 0 else None
        self._f_proj = _Folded(self.proj)

    def pre(self, x, g, out=None, slot: Optional[int] = None, valid_len: Optional[torch.Tensor] = None):
        """``conv_pre(x)`` and ``cond(g)`` (:428, :430): the part of forward that does not need the pitch hidden state,
        so ``Vocoder`` can run it beside the SourceNetwork.  ``out`` = (xp, cg) preallocated by the caller."""
        x, g = _as_input(x), _as_input(g)
        xp = _dense_conv(x, self._f_pre, 7, slot=slot, out=None if out is None else out[0], valid_len=valid_len)
        cg = ops.conv1d_direct(g, self._f_cond.weight(), self._f_cond.bias(), out=None if out is None else out[1])
        return xp, cg

    def forward(self, x, pitch, g=None, _pre=None, *, lengths=None, _table=None):
        """``lengths`` (frames of x per utterance: int CUDA tensor [B] or host sequence): a padded batch of utterances
        of different lengths (pitch: the SourceNetwork's hidden state of the same batch); item b's waveform below
        prod(upsample_rates) * lengths[b] equals its own unpadded run, the rest is 0.  ``_table``: the length table
        ``vocode`` already built for ``_pre``."""
        x, pitch = _as_input(x), _as_input(pitch)
        if g is None:
            # the reference evaluates self.cond(g) unconditionally (:430) and fails on g=None
            raise ValueError("Generator.forward needs the speaker embedding g")
        V = _table if _table is not None else self._length_table(lengths, x)
        vl = (lambda i: None) if V is None else (lambda i: V[i])
        xp, cg = self.pre(x, g, valid_len=vl(0)) if _pre is None else _pre
        proj = proj_ready = None
        if self.parallel_blocks and _PRE_OVERLAP[0]:
            # multi-stream mode: proj(pitch) (:437) and the DBlock's residual conv run beside the DBlock's main branch
            # on two of the (idle) resblock streams, each with its stream's workspace slot
            main = torch.cuda.current_stream()
            s0, s1 = _side_streams(x.device, 3)[:2]
            proj = torch.empty(x.shape[0], self.proj.out_channels, pitch.shape[-1], dtype=torch.float32, device=x.device)
            fork, proj_ready = torch.cuda.Event(), torch.cuda.Event()
            fork.record(main)
            s0.wait_event(fork)
            with torch.cuda.stream(s0):
                _dense_conv(pitch, self._f_proj, 7, slot=0, out=proj, valid_len=vl(1))
                proj_ready.record(s0)
            dn = self.downs(pitch, side=(s1, 1), valid_len=vl(0))
        else:
            dn = self.downs(pitch, valid_len=vl(0))
        x = ops.add3_bcast(xp, dn, cg, out=xp)
        sc = 1.0
        for i in range(self.num_upsamples):
            add = None
            if i == 0:
                if proj is None:
                    add = _dense_conv(pitch, self._f_proj, 7, valid_len=vl(1))
                else:
                    torch.cuda.current_stream().wait_event(proj_ready)
                    add = proj
            x = _dense_convT(x, self._f_ups[i], self.ups[i].kernel_size[0], self.upsample_rates[i], add=add,
                             scale=sc, valid_len=vl(i))
            x, sc = self._stage(x, i, separate=i < self.num_upsamples - 1, valid_len=vl(i + 1))
        self.activation_post.check_filters()
        n = self.num_upsamples
        x = ops.act1d(x, *self.activation_post.params(), scale=sc, **_vl(vl(n)))
        return ops.conv1d_direct(x, self._f_post.weight(), None, pad=3, flags=ops.CONV_TANH, **_vl(vl(n)))

    def remove_weight_norm(self):
        for l in self.ups:
            torch.nn.utils.remove_weight_norm(l)
        for l in self.resblocks:
            l.remove_weight_norm()
        self.downs.remove_weight_norm()
        torch.nn.utils.remove_weight_norm(self.conv_pre)
        self._f_pre = _Folded(self.conv_pre)
        self._f_ups = [_Folded(u) for u in self.ups]


# ----------------------------------------------------------------------------------------------
# SpeechSR
# ----------------------------------------------------------------------------------------------
class SpeechSRGenerator(_VocoderBase):
    """speechsr24k/speechsr.py:67-115 (scale 1.5) and speechsr48k/speechsr.py:67-114 (scale 3).

    The reference hard-codes the ratio in ``forward`` (:96); ``upsample_rates`` only sets the loop
    count.  ``scale`` selects the twin."""

    scale = 1.5

    def __init__(self, initial_channel, resblock, resblock_kernel_sizes, resblock_dilation_sizes, upsample_rates,
                 upsample_initial_channel, upsample_kernel_sizes, gin_channels=0):
        super().__init__()
        self.num_kernels = len(resblock_kernel_sizes)
        self.num_upsamples = len(upsample_rates)
        if self.num_upsamples != 1:
            raise NotImplementedError("the reference builds resblocks for exactly one stage (speechsr.py:77)")
        if initial_channel != 1:
            raise NotImplementedError("SpeechSR conv_pre takes the mono waveform (speechsr.py:242)")
        self.conv_pre = _weight_norm(Conv1d(initial_channel, upsample_initial_channel, 7, 1, padding=3))
        self.resblocks = nn.ModuleList()
        ch = upsample_initial_channel
        for k, d in zip(resblock_kernel_sizes, resblock_dilation_sizes):
            self.resblocks.append(AMPBlock0(ch, k, d, activation="snakebeta"))
        self.activation_post = Activation1d(activation=SnakeBeta(ch, alpha_logscale=True))
        self.conv_post = Conv1d(ch, 1, 7, 1, padding=3, bias=False)
        if gin_channels != 0:
            self.cond = nn.Conv1d(gin_channels, upsample_initial_channel, 1)
        self._f_pre = _Folded(self.conv_pre)
        self._f_post = _Folded(self.conv_post)

    def forward(self, x, g=None, *, lengths=None):
        """``lengths`` (input samples per utterance: int CUDA tensor [B] or host sequence): a padded batch of utterances
        of different lengths; item b's output below int(lengths[b] * scale) equals its own unpadded run, the rest is 0."""
        if g is not None:
            raise NotImplementedError("SpeechSR is unconditional in the reference (gin_channels=0)")
        x = _as_input(x)
        L = x.shape[-1]
        ln = _lengths_tensor(lengths, x.shape[0], L, x.device)
        vin = vout = None
        if ln is not None:
            # int(L * 1.5) == (3 L) // 2 and int(L * 3) == 3 L, in integer arithmetic on the device
            vin, vout = ln, (ln * 3 // 2 if self.scale == 1.5 else ln * int(self.scale))
        x = ops.sr_pre_interp(x, self._f_pre.weight(), self._f_pre.bias(), int(L * self.scale),
                              **_vl(None if ln is None else (vin, vout)))
        x, sc = self._stage(x, 0, valid_len=vout)
        self.activation_post.check_filters()
        x = ops.act1d(x, *self.activation_post.params(), scale=sc, **_vl(vout))
        return ops.conv1d_direct(x, self._f_post.weight(), None, pad=3, flags=ops.CONV_TANH, **_vl(vout))

    def _stream_forward(self, win: torch.Tensor, vin: torch.Tensor, vout: torch.Tensor, origin: torch.Tensor):
        """``forward`` of the streaming windows of ``SpeechSRStream``: win fp32 [S, W], item b the window
        win[b, :vin[b]] at the stream origins origin[b] (``ops.sr_pre_interp_stream``).  Returns [S, 1, W * scale];
        outputs of item b below vout[b] away from the window's edges equal those of the whole stream's ``forward``."""
        up, down = ops.SR_RATIOS[self.scale]
        x = ops.sr_pre_interp_stream(win.unsqueeze(1), self._f_pre.weight(), self._f_pre.bias(),
                                     win.shape[-1] * up // down, (vin, vout), origin, (up, down))
        x, sc = self._stage(x, 0, valid_len=vout)
        self.activation_post.check_filters()
        x = ops.act1d(x, *self.activation_post.params(), scale=sc, valid_len=vout)
        return ops.conv1d_direct(x, self._f_post.weight(), None, pad=3, flags=ops.CONV_TANH, valid_len=vout)

    def remove_weight_norm(self):
        for l in self.resblocks:
            l.remove_weight_norm()
        torch.nn.utils.remove_weight_norm(self.conv_pre)
        self._f_pre = _Folded(self.conv_pre)


class SpeechSR24Generator(SpeechSRGenerator):
    scale = 1.5


class SpeechSR48Generator(SpeechSRGenerator):
    scale = 3


class _SpeechSRSynthesizer(nn.Module):
    """SynthesizerTrn of speechsr24k/speechsr.py:215-252 (inference part: ``dec`` only)."""

    _gen_cls = SpeechSR24Generator

    def __init__(self, spec_channels, segment_size, resblock, resblock_kernel_sizes, resblock_dilation_sizes,
                 upsample_rates, upsample_initial_channel, upsample_kernel_sizes, **kwargs):
        super().__init__()
        self.spec_channels = spec_channels
        self.resblock = resblock
        self.resblock_kernel_sizes = resblock_kernel_sizes
        self.resblock_dilation_sizes = resblock_dilation_sizes
        self.upsample_rates = upsample_rates
        self.upsample_initial_channel = upsample_initial_channel
        self.upsample_kernel_sizes = upsample_kernel_sizes
        self.segment_size = segment_size
        self.dec = self._gen_cls(1, resblock, resblock_kernel_sizes, resblock_dilation_sizes, upsample_rates,
                                 upsample_initial_channel, upsample_kernel_sizes)

    def forward(self, x, *, lengths=None):
        return self.dec(x, lengths=lengths)

    @torch.no_grad()
    def infer(self, x, max_len=None):
        return self.dec(x[:, :, :max_len])


class SpeechSR24(_SpeechSRSynthesizer):
    _gen_cls = SpeechSR24Generator


class SpeechSR48(_SpeechSRSynthesizer):
    _gen_cls = SpeechSR48Generator


def vocode(sn: "SourceNetwork", dec: "Generator", z, g, need_pred: bool = False, *, lengths=None):
    """``e, e_ = sn(z, g); return dec(z, e, g), e_`` (hierspeechpp_speechsynthesizer.py:648-649, :697-698).

    In multi-stream mode (``dec.parallel_blocks``) ``dec.conv_pre(z)`` and ``dec.cond(g)``, which do not depend on the
    SourceNetwork, run beside it on their own stream and operand workspace slot; their outputs are allocated on the
    caller's stream.  ``lengths``: frames of z per utterance (see ``Generator.forward``)."""
    if not (dec.parallel_blocks and z.is_cuda and _PRE_OVERLAP[0]):
        e, e_ = sn(z, g, need_pred=need_pred, lengths=lengths)
        return dec(z, e, g=g, lengths=lengths), e_
    z_, g_ = _as_input(z), _as_input(g)
    B, _, T = z_.shape
    V = dec._length_table(lengths, z_)
    c0 = dec.conv_pre.out_channels
    xp = torch.empty(B, c0, T, dtype=torch.float32, device=z_.device)
    cg = torch.empty(B, c0, 1, dtype=torch.float32, device=z_.device)
    main = torch.cuda.current_stream()
    side = _side_streams(z_.device, 1)[0]
    fork, done = torch.cuda.Event(), torch.cuda.Event()
    fork.record(main)
    side.wait_event(fork)
    with torch.cuda.stream(side):
        dec.pre(z_, g_, out=(xp, cg), slot=_PRE_SLOT, valid_len=None if V is None else V[0])
        done.record(side)
    e, e_ = sn(z_, g_, need_pred=need_pred, lengths=None if V is None else V[0])
    main.wait_event(done)
    return dec(z_, e, g=g_, _pre=(xp, cg), _table=V), e_


class Vocoder(nn.Module):
    """The ``sn`` -> ``dec`` pair as ``SynthesizerTrn`` owns it (hierspeechpp_speechsynthesizer.py:624-625,
    648-649): ``forward(z, g)`` returns the 16 kHz waveform [B,1,320*T]."""

    def __init__(self, **cfg):
        super().__init__()
        from .config import HIER_CFG
        c = dict(HIER_CFG)
        c.update(cfg)
        self.dec = Generator(**c)
        self.sn = SourceNetwork(c["upsample_initial_channel"] // 2)

    def forward(self, z, g, lengths=None):
        """``lengths`` (frames of z per utterance: int CUDA tensor [B] or host sequence): a padded batch of utterances of
        different lengths; item b's waveform [:320 * lengths[b]] equals its own unpadded run, the rest is 0."""
        return vocode(self.sn, self.dec, z, g, lengths=lengths)[0]


class VocoderSR(nn.Module):
    """Config #4's timed stage as ONE callable: ``sn`` -> ``dec`` -> SpeechSR (inference_plm.py:176-181) -> optional
    peak-normalised int16 PCM (:183-188), everything enqueued on one stream with no host round trip, so a
    ``CudaGraphRunner`` replays the whole hand-off as one graph and the host only ever sees 2 bytes per output sample.

    The 16 kHz fp32 waveform between the two models is 4 bytes per sample (0.02 % of the stage's traffic) and stays
    in L2; a kernel-level fusion of ``conv_post+tanh`` into SpeechSR's ``conv_pre+interpolate`` would recompute every
    16 kHz sample ~14x (7 taps x 2 source positions) to save that round trip, so the hand-off is fused at the graph
    level, not the kernel level (DESIGN.md §8f3)."""

    def __init__(self, which: int = 24, **cfg):
        super().__init__()
        from .config import SR_CFG
        if which not in (24, 48):
            raise ValueError("which must be 24 or 48")
        self.vocoder = Vocoder(**cfg)
        self.sr = (SpeechSR24 if which == 24 else SpeechSR48)(100, 40, **SR_CFG)
        self.which = which

    def forward(self, z, g, pcm16: bool = False, lengths=None):
        """``lengths``: frames of z per utterance (see ``Vocoder.forward``); the padding of each output row is 0, which
        leaves its per-utterance PCM peak unchanged."""
        wav16 = self.vocoder(z, g, lengths=lengths)
        hop = _hops(self.vocoder.dec.upsample_rates)[-1]
        out = self.sr(wav16, lengths=_scale_lengths(lengths, hop))
        if pcm16:
            from .runtime import to_pcm16
            return to_pcm16(out, per_utterance=True)
        return out
