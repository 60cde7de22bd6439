"""The step BEFORE the vocoder (SURVEY.md §8f2), B200-native: ``StyleEncoder`` (styleencoder.py:33-99),
``PosteriorSFEncoder`` (hierspeechpp_speechsynthesizer.py:168-203, three ``modules.WN`` stacks) and the reverse pass of
``ResidualCouplingBlock_Transformer`` (:53-88; ``ResidualCouplingLayer_Transformer_simple`` / ``DiTConVBlock`` /
``FFN_Conv`` of modules.py:350-488, timm 0.6.13 ``Attention``).

Same class names, constructor signatures, forward signatures and ``state_dict`` keys as the reference, so the
reference's own ``SynthesizerTrn`` builds them after ``patch_reference()`` and its checkpoints load strictly.  With the
vocoder at ~1 ms these 50 Hz modules are the tail of ``voice_conversion_noise_control`` (:675-699) when run as ~500
eager ATen launches; here every Conv1d / Linear runs on the tcgen05 conv kernel (fp16 operands, fp32 accumulate: the
front is two orders of magnitude less sensitive than the bar, DESIGN.md §8f2) and every other reference expression is
ONE fused launch (csrc/frame_ops.cu), so the whole call replays as one CUDA graph.

Inference only (``reverse=True`` for the flows, eval-mode dropout).  CUDA tensors only; the random draws use
``torch.randn_like`` exactly where the reference does, so a seeded run reproduces the reference's noise."""
from __future__ import annotations

import math
import numbers
from typing import Optional

import torch
from torch import nn
from torch.nn import Conv1d

from . import ops
from .modules import (_Folded, _as_input, _bump_on_load, _frame_mask, _lengths_tensor, _row_tiles, _side_streams,
                      _vl, _weight_norm, Generator, SourceNetwork, vocode)

_S_X, _S_G, _S_W = 4, 5, 6      # blk16 workspace slots of this module family (0..3 and 7 belong to the vocoder)
_WN_TAIL = __import__("os").environ.get("HSV_WN_TAIL", "1") != "0"   # A/B switch: WN layer tail in the res_skip conv's epilogue
_S_X2, _S_G2 = 10, 11           # ... of the second WaveNet stack when two run side by side (8, 9: tests)


class _FoldedLinear(_Folded):
    """nn.Linear as a 1x1 convolution: weight [out, in] -> [out, in, 1]."""

    def __init__(self, lin: nn.Linear):
        super().__init__(lin)

    def weight(self):
        w = self.conv.weight
        key = (w.data_ptr(), w._version, _epoch())
        if key != self.key:
            self.w = w.detach().unsqueeze(-1).contiguous()
            self.packed = None
            self.key = key
        return self.w


def _epoch():
    from . import modules as M
    return M._CACHE_EPOCH[0]


class _FoldedGate(_Folded):
    """A WN in_layer (2H output channels: tanh half | sigmoid half) with its output channels in the order the
    operand-writing gate epilogue wants (``ops.gate_permutation``): weight, bias and packed operand all permuted."""

    def __init__(self, conv, blocks: int = 1):
        super().__init__(conv)
        self.blocks = blocks            # cond_layer: n_layers blocks of 2H channels, each permuted on its own
        self._pkey, self._wperm, self._bperm = None, None, None

    def _perm(self, cout, device):
        per = cout // self.blocks
        base = ops.gate_permutation(per, device)
        return torch.cat([base + i * per for i in range(self.blocks)])

    def weight(self):
        w = _Folded.weight(self)
        if self._pkey != self.key:
            perm = self._perm(w.shape[0], w.device)
            self._wperm = w[perm].contiguous()
            b = _Folded.bias(self)
            self._bperm = None if b is None else b[perm].contiguous()
            self._pkey = self.key
            if w.is_cuda:
                ops._static_data_barrier("WN gate-order weights")
        return self._wperm

    def bias(self):
        self.weight()
        return self._bperm


class _FoldedCat:
    """Several nn.Linear layers with the same input, concatenated along the output dimension (one launch for all)."""

    def __init__(self, lins):
        self.lins = list(lins)
        self.key, self.w, self.b = None, None, None

    def _refresh(self):
        key = tuple((l.weight.data_ptr(), l.weight._version, l.bias.data_ptr(), l.bias._version) for l in self.lins) \
            + (_epoch(),)
        if key != self.key:
            self.w = torch.cat([l.weight.detach() for l in self.lins], 0).unsqueeze(-1).contiguous()
            self.b = torch.cat([l.bias.detach() for l in self.lins], 0).contiguous()
            self.key = key

    def weight(self):
        self._refresh()
        return self.w

    def bias(self):
        self._refresh()
        return self.b


def _mask2d(x_mask: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    if x_mask is None:
        return None
    return _as_input(x_mask.to(torch.float32)).reshape(x_mask.shape[0], -1)


def _conv_buf(buf: torch.Tensor, f: _Folded, L: int, cin: int, cout: int, k: int = 1, d: int = 1) -> torch.Tensor:
    """tcgen05 'same' conv of an already packed operand."""
    B = buf.shape[0]
    wp, nt = f.packed_weight(_row_tiles(B, L))
    return ops.conv1d_umma(buf, wp, f.bias(), L, cin, cout, k, d, nt)


class _FoldedSlice:
    """Input-channel slice [lo, hi) of a folded conv weight, packed on its own (split-K passes of wide layers)."""

    def __init__(self, parent: _Folded, lo: int, hi: int):
        self.parent, self.lo, self.hi = parent, lo, hi
        self.key, self.packed = None, {}

    def packed_weight(self, row_tiles: int):
        w = self.parent.weight()
        key = (w.data_ptr(), self.parent.key)
        if key != self.key:
            self.packed, self.key = {}, key
        nt = ops.pick_n_tile(w.shape[0], row_tiles, (self.hi - self.lo) * w.shape[2])
        if nt not in self.packed:
            self.packed[nt] = ops.pack_conv_weight(w[:, self.lo:self.hi].contiguous(), nt)
        return self.packed[nt], nt


def _conv(x: torch.Tensor, f: _Folded, k: int = 1, d: int = 1, mode: int = ops.PACK_MASK, C: Optional[int] = None,
          slot: int = _S_X, mask=None, bcast=None, strided: bool = False) -> torch.Tensor:
    """pack (with a fused activation) -> tcgen05 conv.  ``C`` = operand channels when x is wider (prefix / gate).

    The tcgen05 kernel keeps the whole [128 x Cin] operand tile in shared memory (Cin <= 512): wider layers
    (pre_source 1024 -> 192, FFN fc2 768 -> 192) run as split-K passes over input-channel slices, each pass adding
    the previous result in its epilogue (fp32).  ``strided``: at any batch size, ONE pack of all channels and passes
    that read its channel ranges in place (the launches of the batch-1 path; per-item batches use it)."""
    B, cx, L = x.shape
    C = cx if C is None else C
    cout = f.conv.out_channels if hasattr(f.conv, "out_channels") else f.conv.out_features
    if C <= 512:
        buf = ops.blk16_buffer(B, C, L, x.device, slot)
        ops.pack_blk16_act(x, buf, C, mode, bcast=bcast, mask=mask)
        ops.check_saturation(buf, C, L)
        return _conv_buf(buf, f, L, C, cout, k, d)
    if mode == ops.PACK_GATE:
        raise NotImplementedError("split-K: the gate packer reads two channel halves")
    nsplit = (C + 511) // 512
    per = C // nsplit
    if per * nsplit != C or per % 16:
        raise NotImplementedError(f"split-K: Cin={C} does not split into equal multiples of 16")
    if not hasattr(f, "_slices") or f._slices[0] != (C, nsplit):
        f._slices = ((C, nsplit), [_FoldedSlice(f, i * per, (i + 1) * per) for i in range(nsplit)])
    out = None
    whole = None
    if (B == 1 or strided) and per % ops.blk_cw(C) == 0 and ops.blk_cw(per) == ops.blk_cw(C):
        # one batch item: the channel chunks of a blk16 buffer are its outermost dimension, so ONE pack of all C channels
        # serves every pass as a dense sub-buffer
        whole = ops.blk16_buffer(B, C, L, x.device, slot)
        ops.pack_blk16_act(x, whole, C, mode, mask=mask)
        ops.check_saturation(whole, C, L)
        nchunk = whole.shape[1] * per // C            # channel chunks per pass
    for i, fs in enumerate(f._slices[1]):
        if whole is not None:
            buf = whole[:, i * nchunk:(i + 1) * nchunk]
        else:
            buf = ops.blk16_buffer(B, per, L, x.device, slot)
            ops.pack_blk16_act(x, buf, per, mode, mask=mask, c_off=i * per)
            ops.check_saturation(buf, per, L)
        wp, nt = fs.packed_weight(_row_tiles(B, L))
        out = ops.conv1d_umma(buf, wp, f.bias() if i == 0 else None, L, per, cout, k, d, nt, residual=out)
    return out


def _slices_of(f: _Folded, C: int):
    nsplit = (C + 511) // 512
    per = C // nsplit
    if per * nsplit != C or per % 16:
        raise NotImplementedError(f"split-K: Cin={C} does not split into equal multiples of 16")
    if not hasattr(f, "_slices") or f._slices[0] != (C, nsplit):
        f._slices = ((C, nsplit), [_FoldedSlice(f, i * per, (i + 1) * per) for i in range(nsplit)])
    return per, f._slices[1]


def _conv_packed(buf: torch.Tensor, f: _Folded, C: int, L: int, k: int = 1, d: int = 1,
                 strided: bool = False) -> torch.Tensor:
    """tcgen05 conv of an already packed operand of C channels; wider than 512: split-K over channel sub-buffers
    (batch 1, where the channel chunks are the outermost dimension of the buffer, or ``strided``: the passes read
    the channel ranges in place through the operand's batch stride)."""
    B = buf.shape[0]
    cout = f.conv.out_channels if hasattr(f.conv, "out_channels") else f.conv.out_features
    if C <= 512:
        return _conv_buf(buf, f, L, C, cout, k, d)
    if B != 1 and not strided:
        raise NotImplementedError("split-K over a packed buffer needs batch 1 or strided=True")
    per, slices = _slices_of(f, C)
    nchunk = buf.shape[1] * per // C
    out = None
    for i, fs in enumerate(slices):
        wp, nt = fs.packed_weight(_row_tiles(B, L))
        out = ops.conv1d_umma(buf[:, i * nchunk:(i + 1) * nchunk], wp, f.bias() if i == 0 else None, L, per, cout, k, d, nt,
                              residual=out)
    return out


def _vec(x: torch.Tensor, f: _Folded, silu: bool = False) -> torch.Tensor:
    """Linear / 1x1 conv on a per-utterance vector [B, Cin] -> [B, Cout] (fp32 warp-per-output dot products)."""
    B = x.shape[0]
    y = ops.conv1d_direct(x.reshape(B, -1, 1).contiguous(), f.weight(), f.bias(), flags=ops.CONV_SILU_IN if silu else 0)
    return y.view(B, -1)


# ----------------------------------------------------------------------------------------------
# modules.WN  (modules.py:111-182)
# ----------------------------------------------------------------------------------------------
class WN(nn.Module):
    def __init__(self, hidden_channels, kernel_size, dilation_rate, n_layers, gin_channels=0, p_dropout=0):
        super().__init__()
        assert kernel_size % 2 == 1
        self.hidden_channels = hidden_channels
        self.kernel_size = (kernel_size,)
        self.dilation_rate = dilation_rate
        self.n_layers = n_layers
        self.gin_channels = gin_channels
        self.p_dropout = p_dropout
        self.in_layers = nn.ModuleList()
        self.res_skip_layers = nn.ModuleList()
        self.drop = nn.Dropout(p_dropout)
        if gin_channels != 0:
            self.cond_layer = _weight_norm(Conv1d(gin_channels, 2 * hidden_channels * n_layers, 1))
        for i in range(n_layers):
            dilation = dilation_rate ** i
            padding = int((kernel_size * dilation - dilation) / 2)
            self.in_layers.append(_weight_norm(Conv1d(hidden_channels, 2 * hidden_channels, kernel_size,
                                                      dilation=dilation, padding=padding)))
            rs = 2 * hidden_channels if i < n_layers - 1 else hidden_channels
            self.res_skip_layers.append(_weight_norm(Conv1d(hidden_channels, rs, 1)))
        self._refold()
        _bump_on_load(self)

    def _refold(self):
        # in_layers / cond_layer in gate order: the in_layer conv's epilogue evaluates the gate and writes the
        # res_skip conv's fp16 operand directly (csrc/conv_umma.cu, hsv_conv1d_umma_blk16)
        self._f_in = [_FoldedGate(c) for c in self.in_layers]
        self._f_rs = [_Folded(c) for c in self.res_skip_layers]
        self._f_cond = _FoldedGate(self.cond_layer, blocks=self.n_layers) if self.gin_channels != 0 else None

    def forward(self, x, x_mask, g=None, slots=(_S_X, _S_G), **kwargs):
        """``slots``: the two operand workspace slots of this call (two WN stacks on two streams need two pairs)."""
        x = _as_input(x)
        mask = _mask2d(x_mask)
        B, H, T = x.shape
        k = self.kernel_size[0]
        n = self.n_layers
        sx, sg = slots
        gl = None
        if g is not None:
            # cond_layer(g): [B, n, 2H] (each layer's 2H block in gate order); a layer's slice is a strided row view
            gl = _vec(_as_input(g).reshape(B, -1), self._f_cond).view(B, n, 2 * H)
        x = x.clone()
        output = torch.zeros_like(x)
        # the operand of in_layers[0]; every later layer's operand is written by the previous layer's fused tail
        buf = ops.blk16_buffer(B, H, T, x.device, sx)
        gbuf = ops.blk16_buffer(B, H, T, x.device, sg)
        ops.pack_blk16_act(x, buf, H, ops.PACK_MASK)
        ops.check_saturation(buf, H, T)
        rt = _row_tiles(B, T)
        for i in range(n):
            d = self.dilation_rate ** i
            # in_layers[i] -> + cond -> tanh * sigmoid, straight into the res_skip conv's operand
            wp, nt = self._f_in[i].packed_weight(rt)
            ops.conv1d_umma_blk(buf, wp, self._f_in[i].bias(), T, H, 2 * H, k, d, nt, gbuf, ops.BLK_GATE,
                                bc=None if gl is None else gl[:, i])
            ops.check_saturation(gbuf, H, T)
            if i < n - 1:
                # res_skip conv with the layer tail in its epilogue: x = (x + res) * mask, output += skip (both in place),
                # buf = fp16(x) = the next in_layer's operand
                wr, ntr = self._f_rs[i].packed_weight(rt)
                if H % ntr == 0 and _WN_TAIL:
                    ops.conv1d_umma_wn_tail(gbuf, wr, self._f_rs[i].bias(), x, output, mask, buf, ntr)
                else:
                    acts_rs = ops.conv1d_umma(gbuf, wr, self._f_rs[i].bias(), T, H, 2 * H, 1, 1, ntr)
                    ops.wn_res_pack(x, acts_rs, mask, output, buf)
                ops.check_saturation(buf, H, T)
            else:
                acts_rs = _conv_buf(gbuf, self._f_rs[i], T, H, H)
                ops.frame_op(ops.OP_WN_LAST, None, acts_rs, None, mask, None, output, B, H, T)
        return output

    def remove_weight_norm(self):
        if self.gin_channels != 0:
            torch.nn.utils.remove_weight_norm(self.cond_layer)
        for l in list(self.in_layers) + list(self.res_skip_layers):
            torch.nn.utils.remove_weight_norm(l)
        self._refold()


# ----------------------------------------------------------------------------------------------
# PosteriorSFEncoder  (hierspeechpp_speechsynthesizer.py:168-203)
# ----------------------------------------------------------------------------------------------
class PosteriorSFEncoder(nn.Module):
    parallel_blocks = False     # multi-stream mode (set together with the vocoder's switch)

    def __init__(self, src_channels, out_channels, hidden_channels, kernel_size, dilation_rate, n_layers,
                 gin_channels=0):
        super().__init__()
        self.out_channels = out_channels
        self.hidden_channels = hidden_channels
        self.kernel_size = kernel_size
        self.dilation_rate = dilation_rate
        self.n_layers = n_layers
        self.gin_channels = gin_channels
        self.pre_source = nn.Conv1d(src_channels, hidden_channels, 1)
        self.pre_filter = nn.Conv1d(1, hidden_channels, kernel_size=9, stride=4, padding=4)
        self.source_enc = WN(hidden_channels, kernel_size, dilation_rate, n_layers // 2, gin_channels=gin_channels)
        self.filter_enc = WN(hidden_channels, kernel_size, dilation_rate, n_layers // 2, gin_channels=gin_channels)
        self.enc = WN(hidden_channels, kernel_size, dilation_rate, n_layers // 2, gin_channels=gin_channels)
        self.proj = nn.Conv1d(hidden_channels, out_channels * 2, 1)
        self._f_src = _Folded(self.pre_source)
        self._f_proj = _Folded(self.proj)
        _bump_on_load(self)

    def forward(self, x_src, x_ftr, x_mask, g=None, *, eps=None, noise_scale=1.0, lengths=None, seed=None):
        """``eps``: the noise of z = (m + eps * exp(logs) * noise_scale) * mask, fp32 [B, out_channels, T] (default: one
        ``torch.randn_like(m)`` draw, the reference's :201).  ``lengths`` (frames per item: int CUDA tensor [B] or host
        sequence): a padded batch whose item b equals its own unpadded run with ``x_mask`` = ones (f0 past
        4 * lengths[b] is never read, nor is any other input past the item); ``x_mask`` is then derived from them.
        With ``lengths`` only: ``seed`` (int64 CUDA tensor [B] or host sequence; not with ``eps``) generates item b's noise
        from seed[b] inside the sampling launch, equal to ``eps = ops.seeded_normal(seed[b:b+1], out_channels, len[b])``;
        ``noise_scale`` may be a floating CUDA tensor [B] (item b as with ``float(noise_scale[b])``)."""
        B, _, T = x_src.shape
        vl = _lengths_tensor(lengths, B, T, x_src.device)
        seeds = _per_item_noise_args(vl is not None, B, x_src.device, eps, seed, noise_scale=noise_scale)
        x_src, x_ftr = _as_input(x_src), _as_input(x_ftr)
        if vl is not None:
            x_mask = _frame_mask(vl, T).unsqueeze(1)
        mask = _mask2d(x_mask)
        H = self.hidden_channels
        if vl is None:
            xs = _conv(x_src, self._f_src)
        else:   # the batch-1 split-K launches at every B; padding never enters the operand
            xs = _conv(x_src, self._f_src, mask=mask, strided=True)
        ops.frame_op(ops.OP_MASK, xs, None, None, mask, xs, None, B, H, T)
        xf = ops.conv1d_c1_strided(x_ftr, self.pre_filter.weight.detach(), self.pre_filter.bias.detach(), 4, 4, mask,
                                   **_vl(vl))
        if xf.shape[-1] != T:
            raise ValueError(f"f0 has {x_ftr.shape[-1]} frames, expected 4 x {T}")
        if self.parallel_blocks:
            # the two WaveNet stacks are independent (:197-198): second stream, second pair of workspace slots
            main = torch.cuda.current_stream()
            side = _side_streams(xs.device, 3)[0]
            fork, done = torch.cuda.Event(), torch.cuda.Event()
            fork.record(main)
            side.wait_event(fork)
            with torch.cuda.stream(side):
                xf = self.filter_enc(xf, x_mask, g=g, slots=(_S_X2, _S_G2))
                done.record(side)
            xs = self.source_enc(xs, x_mask, g=g)
            main.wait_event(done)
        else:
            xs = self.source_enc(xs, x_mask, g=g)
            xf = self.filter_enc(xf, x_mask, g=g)
        ops.frame_op(ops.OP_ADD, xs, xf, None, None, xs, None, B, H, T)
        x = self.enc(xs, x_mask, g=g)
        stats = _conv(x, self._f_proj)
        ops.frame_op(ops.OP_MASK, stats, None, None, mask, stats, None, B, 2 * self.out_channels, T)
        m, logs = torch.split(stats, self.out_channels, dim=1)
        per_item_ns = vl is not None and _per_item_control(noise_scale, B, stats.device)
        if seeds is not None or per_item_ns:
            if eps is not None:
                _check_eps(eps, B, self.out_channels, T, stats.device)
            elif seeds is None:
                eps = torch.randn_like(m)
            ns = noise_scale.to(torch.float32).contiguous() if per_item_ns else float(noise_scale)
            z = ops.sample_ragged(stats, ns, vl, eps=None if eps is None else eps.contiguous(), seeds=seeds)
            return z, m, logs
        if eps is None:
            eps = torch.randn_like(m)                  # the reference's draw (:201), same generator, same shape
        else:
            _check_eps(eps, B, self.out_channels, T, stats.device)
        z = torch.empty(B, self.out_channels, T, dtype=torch.float32, device=stats.device)
        ops.frame_op(ops.OP_SAMPLE, stats, eps.contiguous(), None, mask, z, None, B, self.out_channels, T,
                     s=float(noise_scale))
        return z, m, logs


def _seeds_tensor(seed, B: int, device) -> torch.Tensor:
    """Per-item seeds as a contiguous int64 [B] tensor on ``device``: an int64 tensor there is only checked (never read
    back, so the call stays capturable); a host sequence of ints in the int64 range is copied."""
    device = torch.device(device)
    if isinstance(seed, torch.Tensor):
        if seed.device != device:
            raise ValueError(f"seed is on {seed.device}, the input is on {device}")
        if tuple(seed.shape) != (B,) or seed.dtype != torch.int64:
            raise ValueError(f"seed must be an int64 tensor of shape ({B},), got {seed.dtype} {tuple(seed.shape)}")
        return seed.contiguous()
    try:
        if isinstance(seed, (str, bytes)):
            raise TypeError
        vals = list(seed)
    except TypeError:
        raise ValueError("seed must be a tensor or a sequence with one seed per item") from None
    if len(vals) != B:
        raise ValueError(f"seed has {len(vals)} entries for a batch of {B}")
    if any(not isinstance(v, numbers.Integral) for v in vals):
        raise ValueError("seeds must be integers")
    vals = [int(v) for v in vals]
    if any(not -(1 << 63) <= v < (1 << 63) for v in vals):
        raise ValueError("seeds must lie in the int64 range")
    return torch.tensor(vals, dtype=torch.int64, device=device)


def _per_item_control(v, B: int, device) -> bool:
    """noise_scale / denoise_ratio of a per-item call: a floating tensor of shape (B,) on the input's device holds one
    value per item; a Python number or any other one-element tensor is one value for the whole call, as before."""
    return (isinstance(v, torch.Tensor) and v.is_floating_point() and tuple(v.shape) == (B,)
            and v.device == torch.device(device))


def _per_item_noise_args(per_item: bool, B: int, device, eps, seed, **controls) -> Optional[torch.Tensor]:
    """Checks ``seed`` and the controls of a call (a tensor of more than one element is per item: per-item calls only,
    and there a floating [B] tensor on the input's device); returns the int64 seeds or None."""
    multi = [k for k, v in controls.items() if isinstance(v, torch.Tensor) and v.numel() > 1]
    if not per_item and (seed is not None or multi):
        what = ", ".join((["seed"] if seed is not None else []) + [f"a tensor {k} of several values" for k in multi])
        raise ValueError(f"{what}: per-item batches only (per_item=True / lengths=)")
    if seed is not None and eps is not None:
        raise ValueError("seed= and eps= are exclusive: the seed generates the noise eps would give")
    for k, v in controls.items():
        if isinstance(v, torch.Tensor) and v.numel() > 1 and not _per_item_control(v, B, device):
            raise ValueError(f"{k} must be a float, a one-element tensor or a floating tensor of shape ({B},) on "
                             f"{device}, got {v.dtype} {tuple(v.shape)} on {v.device}")
    return None if seed is None else _seeds_tensor(seed, B, device)


def _check_eps(eps, B: int, C: int, T: int, device):
    if not isinstance(eps, torch.Tensor) or eps.dtype != torch.float32 or eps.device != torch.device(device):
        raise ValueError(f"eps must be a float32 tensor on {device}")
    if tuple(eps.shape) != (B, C, T):
        raise ValueError(f"eps must have shape {(B, C, T)}, got {tuple(eps.shape)}")


# ----------------------------------------------------------------------------------------------
# DiT coupling flows  (modules.py:350-488)
# ----------------------------------------------------------------------------------------------
class Attention(nn.Module):
    """timm 0.6.13 ``vision_transformer.Attention`` (requirements.txt:10): parameter holder + fused forward on
    channel-major [B, C, T] tensors (the reference transposes to [B, T, C] around it)."""

    def __init__(self, dim, num_heads=8, qkv_bias=False, attn_drop=0., proj_drop=0.):
        super().__init__()
        assert dim % num_heads == 0
        self.num_heads = num_heads
        self.scale = (dim // num_heads) ** -0.5
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(proj_drop)
        self._f_qkv = _FoldedLinear(self.qkv)
        self._f_proj = _FoldedLinear(self.proj)

    def run(self, buf: torch.Tensor, C: int, T: int, vl: Optional[torch.Tensor] = None) -> torch.Tensor:
        """buf = packed (normalised, modulated) input; returns proj(attention) fp32 [B, C, T].  ``vl``: per-item lengths
        (int32 [B]): item b attends over its own frames only, as its own run does."""
        B = buf.shape[0]
        qkv = _conv_buf(buf, self._f_qkv, T, C, 3 * C)
        D = C // self.num_heads
        flat = qkv.view(-1)
        if vl is not None and not (ops.MHA_VARIANT[0] == 0 and D in (64, 96, 128)):
            raise NotImplementedError("per-item lengths need the tensor-core attention (head dim 64, 96 or 128)")
        if ops.MHA_VARIANT[0] == 0 and D in (64, 96, 128):
            # the tensor-core attention writes the proj conv's fp16 operand directly
            ab = ops.mha(flat, flat[C * T:], flat[2 * C * T:], B, self.num_heads, D, T, T, 3 * C * T, 3 * C * T, 3 * C * T,
                         self.scale, prescale_q=False, out_blk=ops.blk16_buffer(B, C, T, qkv.device, _S_G), **_vl(vl))
            ops.check_saturation(ab, C, T)
            return _conv_buf(ab, self._f_proj, T, C, C)
        att = ops.mha(flat, flat[C * T:], flat[2 * C * T:], B, self.num_heads, D, T, T, 3 * C * T, 3 * C * T, 3 * C * T,
                      self.scale, prescale_q=False)
        return _conv(att, self._f_proj, slot=_S_G)


class FFN_Conv(nn.Module):
    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, norm_layer=None,
                 bias=True, kernel=5, p_dropout=0.1):
        super().__init__()
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        self.fc1 = nn.Conv1d(in_features, hidden_features, kernel_size=kernel, stride=1, padding=(kernel - 1) // 2,
                             bias=bias)
        self.act = act_layer()
        self.norm = nn.Identity()
        self.fc2 = nn.Conv1d(hidden_features, out_features, kernel_size=1, bias=bias)
        self.drop = nn.Dropout(p_dropout)
        self.kernel = kernel
        self._f1, self._f2 = _Folded(self.fc1), _Folded(self.fc2)

    def run(self, buf: torch.Tensor, C: int, T: int, mask, per_item: bool = False) -> torch.Tensor:
        """fc2(gelu(fc1(buf)) * mask); the trailing * mask is the caller's.  ``per_item``: the batch-1 launches at any
        batch size (a per-item batch must compute what each item's own run computes)."""
        B = buf.shape[0]
        Hh = self.fc1.out_channels
        if B == 1 or Hh <= 512 or per_item:
            # fc1's epilogue applies GELU * mask and writes fc2's fp16 operand; fc2 wider than 512 input channels runs as
            # split-K passes over channel sub-buffers (dense at batch 1, read in place through the batch stride else)
            hb = ops.blk16_buffer(B, Hh, T, buf.device, _S_W)
            wp, nt = self._f1.packed_weight(_row_tiles(B, T))
            ops.conv1d_umma_blk(buf, wp, self._f1.bias(), T, C, Hh, self.kernel, 1, nt, hb, ops.BLK_GELU, mask=mask)
            ops.check_saturation(hb, Hh, T)
            return _conv_packed(hb, self._f2, Hh, T, strided=per_item)
        h = _conv_buf(buf, self._f1, T, C, Hh, self.kernel, 1)
        return _conv(h, self._f2, mode=ops.PACK_GELU, slot=_S_W, mask=mask)


class DiTConVBlock(nn.Module):
    def __init__(self, hidden_size, num_heads, mlp_ratio=4.0, kernel=9, p_dropout=0.1, **block_kwargs):
        super().__init__()
        self.hidden_size = hidden_size
        self.norm1 = nn.LayerNorm(hidden_size, elementwise_affine=False, eps=1e-6)
        self.attn = Attention(hidden_size, num_heads=num_heads, qkv_bias=True, **block_kwargs)
        self.norm2 = nn.LayerNorm(hidden_size, elementwise_affine=False, eps=1e-6)
        self.mlp = FFN_Conv(in_features=hidden_size, hidden_features=int(hidden_size * mlp_ratio),
                            act_layer=lambda: nn.GELU(approximate="tanh"), kernel=kernel, p_dropout=p_dropout)
        self.adaLN_modulation = nn.Sequential(nn.SiLU(), nn.Linear(hidden_size, 6 * hidden_size, bias=True))
        self._f_ada = _FoldedLinear(self.adaLN_modulation[1])

    def run(self, x: torch.Tensor, c: torch.Tensor, mask, mod: Optional[torch.Tensor] = None,
            masked_input: bool = False, pending=None, defer: bool = False, vl: Optional[torch.Tensor] = None):
        """x fp32 [B, C, T] (updated in place), c [B, C] conditioning, mask [B, T] or None.  Returns (x, pending).

        ``mod``: this block's adaLN vector [B, 6C] (rows may be strided) when the caller evaluated all blocks'
        modulations in one launch; ``masked_input``: x is already x * mask (the output of a previous block:
        x*m + g*y*m re-masked is the same bits), so the leading mask pass is skipped.  Every gated residual update
        ``x += gate * y * mask`` (:408-409) is fused into the LayerNorm/modulate/pack launch that follows it:
        ``pending`` = the (y, gate) of the previous block's MLP branch still to be applied, ``defer`` = hand this block's
        own last update to the next block the same way instead of applying it here.  ``vl``: per-item lengths (int32 [B],
        ``mask`` their frame mask): attention over each item's own frames, fc1's operand zero past them."""
        B, C, T = x.shape
        if mask is not None and not masked_input:
            ops.frame_op(ops.OP_MASK, x, None, None, mask, x, None, B, C, T)
        if mod is None:
            mod = _vec(c, self._f_ada, silu=True)                  # [B, 6C]: shift/scale/gate msa, shift/scale/gate mlp
        ms = mod.stride(0)
        sh1, sc1, g1, sh2, sc2, g2 = (mod[:, i * C:(i + 1) * C] for i in range(6))
        buf = ops.blk16_buffer(B, C, T, x.device, _S_X)
        if pending is None:
            ops.ln_mod_blk16(x, sh1, sc1, buf, ms, mask, 1e-6, premask=True)
        else:
            if pending[1].stride(0) != ms:
                raise RuntimeError("DiTConVBlock: pending gate and this block's modulation must share a batch stride")
            ops.gate_ln_mod_blk16(x, pending[0], pending[1], sh1, sc1, buf, ms, mask, 1e-6, premask=True)
        y = self.attn.run(buf, C, T, vl)
        # per item: fc1 (k = 5) must see the zero padding of each item's own run past its length
        ops.gate_ln_mod_blk16(x, y, g1, sh2, sc2, buf, ms, mask, 1e-6, premask=False,
                              **({} if vl is None else {"zero_masked": True}))
        y = self.mlp.run(buf, C, T, mask, per_item=vl is not None)
        if defer:
            return x, (y, g2)
        ops.frame_op(ops.OP_GATE_ADD, x, y, g2, mask, x, None, B, C, T, cstride=ms)
        return x, None


class ResidualCouplingLayer_Transformer_simple(nn.Module):
    def __init__(self, channels, hidden_channels, kernel_size, dilation_rate, n_layers, p_dropout=0.1, mean_only=False):
        assert channels % 2 == 0
        super().__init__()
        if not mean_only:
            raise NotImplementedError("the reference builds these flows with mean_only=True "
                                      "(hierspeechpp_speechsynthesizer.py:75)")
        self.channels = channels
        self.hidden_channels = hidden_channels
        self.n_layers = n_layers
        self.half_channels = channels // 2
        self.mean_only = mean_only
        self.pre = nn.Conv1d(self.half_channels, hidden_channels, 1)
        self.enc_block = nn.ModuleList([DiTConVBlock(hidden_channels, 2, mlp_ratio=4.0, kernel=5, p_dropout=p_dropout)
                                        for _ in range(n_layers)])
        self.post = nn.Conv1d(hidden_channels, self.half_channels, 1)
        self.post.weight.data.zero_()
        self.post.bias.data.zero_()
        self._f_pre, self._f_post = _Folded(self.pre), _Folded(self.post)
        _bump_on_load(self)

    def forward(self, x, x_mask, g=None, reverse=False, mods=None, *, lengths=None):
        """``mods``: [B, n_layers, 6H] adaLN vectors of this layer's blocks, when the owning
        ``ResidualCouplingBlock_Transformer`` evaluated them for all its flows at once.  ``lengths``: as
        ``ResidualCouplingBlock_Transformer.forward``."""
        if not reverse:
            raise NotImplementedError("inference path: reverse=True only")
        x = _as_input(x)
        vl = _lengths_tensor(lengths, x.shape[0], x.shape[-1], x.device)
        if vl is not None:
            x_mask = _frame_mask(vl, x.shape[-1])
        mask = _mask2d(x_mask)
        B, C, T = x.shape
        half, H = self.half_channels, self.hidden_channels
        h = _conv(x, self._f_pre, C=half)                                   # pre(x0): the first half of the channels
        pending = None
        nb = len(self.enc_block)
        for j, blk in enumerate(self.enc_block):
            h, pending = blk.run(h, g, mask, None if mods is None else mods[:, j], masked_input=j > 0, pending=pending,
                                 defer=j < nb - 1, vl=vl)
        m = _conv(h, self._f_post)
        out = x.clone()
        ops.frame_op(ops.OP_COUPLE, out, m, None, mask, out, None, B, half, T)   # x1 = (x1 - m) * mask
        return out


class Flip(nn.Module):
    def forward(self, x, *args, reverse=False, **kwargs):
        x = _as_input(x)
        B, C, T = x.shape
        out = torch.empty_like(x)
        ops.frame_op(ops.OP_FLIP, x, None, None, None, out, None, B, C, T)
        if not reverse:
            return out, torch.zeros(B, dtype=x.dtype, device=x.device)
        return out


class ResidualCouplingBlock_Transformer(nn.Module):
    def __init__(self, channels, hidden_channels, kernel_size, dilation_rate, n_layers=3, n_flows=4, gin_channels=0):
        super().__init__()
        self.channels = channels
        self.hidden_channels = hidden_channels
        self.n_layers = n_layers
        self.n_flows = n_flows
        self.gin_channels = gin_channels
        self.cond_block = nn.Sequential(nn.Linear(gin_channels, 4 * hidden_channels), nn.SiLU(),
                                        nn.Linear(4 * hidden_channels, hidden_channels))
        self.flows = nn.ModuleList()
        for _ in range(n_flows):
            self.flows.append(ResidualCouplingLayer_Transformer_simple(channels, hidden_channels, kernel_size,
                                                                       dilation_rate, n_layers, mean_only=True))
            self.flows.append(Flip())
        self._f_c0, self._f_c2 = _FoldedLinear(self.cond_block[0]), _FoldedLinear(self.cond_block[2])
        self._f_ada_all = _FoldedCat([blk.adaLN_modulation[1] for i in range(0, 2 * n_flows, 2)
                                      for blk in self.flows[i].enc_block])
        _bump_on_load(self)

    def forward(self, x, x_mask, g=None, reverse=False, *, lengths=None):
        """``lengths`` (frames per item: int CUDA tensor [B] or host sequence): a padded batch whose item b equals its own
        unpadded run (x_mask = ones) bit for bit, with 0 past its length; ``x_mask`` is then derived from them."""
        if not reverse:
            raise NotImplementedError("inference path: reverse=True only")
        B = x.shape[0]
        vl = _lengths_tensor(lengths, B, x.shape[-1], x.device)
        if vl is not None:
            x_mask = _frame_mask(vl, x.shape[-1]).unsqueeze(1)
        c = _vec(_vec(_as_input(g).reshape(B, -1), self._f_c0), self._f_c2, silu=True)
        # every DiT block's adaLN modulation depends on c only: ONE launch for all n_flows * n_layers blocks
        # (concatenated weights, cached per checkpoint) instead of one per block on the critical path
        nl, H = self.n_layers, self.hidden_channels
        mods = _vec(c, self._f_ada_all, silu=True).view(B, self.n_flows, nl, 6 * H)
        for idx in reversed(range(len(self.flows))):
            flow = self.flows[idx]
            if idx % 2 == 0:
                x = flow(x, x_mask, g=c, reverse=True, mods=mods[:, idx // 2], lengths=vl)
            else:
                x = flow(x, x_mask, g=c, reverse=True)
        return x


# ----------------------------------------------------------------------------------------------
# StyleEncoder  (styleencoder.py)
# ----------------------------------------------------------------------------------------------
class Mish(nn.Module):
    def forward(self, x):
        raise RuntimeError("Mish is fused into the operand packers of StyleEncoder on this path")


class Conv1dGLU(nn.Module):
    def __init__(self, in_channels, out_channels, kernel_size, dropout):
        super().__init__()
        self.out_channels = out_channels
        self.conv1 = nn.Conv1d(in_channels, 2 * out_channels, kernel_size=kernel_size, padding=2)
        self.dropout = nn.Dropout(dropout)
        self.kernel_size = kernel_size
        self._f = _Folded(self.conv1)

    def run(self, x, mask):
        B, C, T = x.shape
        y = _conv(x, self._f, self.kernel_size, 1)
        ops.frame_op(ops.OP_GLU_RES, x, y, None, mask, x, None, B, C, T)
        return x


class MultiHeadAttention(nn.Module):
    """attentions.MultiHeadAttention (:109-188) without relative-position / proximal terms (StyleEncoder's use)."""

    def __init__(self, channels, out_channels, n_heads, p_dropout=0., window_size=None, heads_share=True,
                 block_length=None, proximal_bias=False, proximal_init=False):
        super().__init__()
        assert channels % n_heads == 0
        if window_size is not None or block_length is not None or proximal_bias:
            raise NotImplementedError("relative / local / proximal attention is not used on this path")
        self.channels, self.out_channels, self.n_heads = channels, out_channels, n_heads
        self.k_channels = channels // n_heads
        self.conv_q = nn.Conv1d(channels, channels, 1)
        self.conv_k = nn.Conv1d(channels, channels, 1)
        self.conv_v = nn.Conv1d(channels, channels, 1)
        self.conv_o = nn.Conv1d(channels, out_channels, 1)
        self.drop = nn.Dropout(p_dropout)
        nn.init.xavier_uniform_(self.conv_q.weight)
        nn.init.xavier_uniform_(self.conv_k.weight)
        nn.init.xavier_uniform_(self.conv_v.weight)
        if proximal_init:
            with torch.no_grad():
                self.conv_k.weight.copy_(self.conv_q.weight)
                self.conv_k.bias.copy_(self.conv_q.bias)
        self._fq, self._fk, self._fv, self._fo = (_Folded(c) for c in (self.conv_q, self.conv_k, self.conv_v, self.conv_o))

    def run(self, x, lens, vl: Optional[torch.Tensor] = None):
        """``lens``: the reference's masked_fill(-1e4) over the padded length; ``vl`` instead: per-item lengths, each
        item attending over its own frames only, as its own run does."""
        B, C, T = x.shape
        buf = ops.blk16_buffer(B, C, T, x.device, _S_X)
        ops.pack_blk16_act(x, buf, C, ops.PACK_MASK)
        q, k, v = (_conv_buf(buf, f, T, C, C) for f in (self._fq, self._fk, self._fv))
        att = ops.mha(q, k, v, B, self.n_heads, self.k_channels, T, T, C * T, C * T, C * T,
                      1.0 / math.sqrt(self.k_channels), prescale_q=True, lens=lens, **_vl(vl))
        return _conv(att, self._fo, slot=_S_G)


class StyleEncoder(nn.Module):
    def __init__(self, in_dim=513, hidden_dim=128, out_dim=256):
        super().__init__()
        self.in_dim, self.hidden_dim, self.out_dim = in_dim, hidden_dim, out_dim
        self.kernel_size, self.n_head, self.dropout = 5, 2, 0.1
        self.spectral = nn.Sequential(nn.Conv1d(in_dim, hidden_dim, 1), Mish(), nn.Dropout(self.dropout),
                                      nn.Conv1d(hidden_dim, hidden_dim, 1), Mish(), nn.Dropout(self.dropout))
        self.temporal = nn.Sequential(Conv1dGLU(hidden_dim, hidden_dim, self.kernel_size, self.dropout),
                                      Conv1dGLU(hidden_dim, hidden_dim, self.kernel_size, self.dropout))
        self.slf_attn = MultiHeadAttention(hidden_dim, hidden_dim, self.n_head, p_dropout=self.dropout,
                                           proximal_bias=False, proximal_init=True)
        self.atten_drop = nn.Dropout(self.dropout)
        self.fc = nn.Conv1d(hidden_dim, out_dim, 1)
        self._f_s0, self._f_s3, self._f_fc = _Folded(self.spectral[0]), _Folded(self.spectral[3]), _Folded(self.fc)
        _bump_on_load(self)

    def forward(self, x, mask=None, *, lengths=None):
        """``lengths`` (frames per item: int CUDA tensor [B] or host sequence): a padded batch whose item b equals, bit for
        bit, its own unpadded run (mask = ones); ``mask`` is then derived from them and x past an item is never used."""
        x = _as_input(x)
        B, _, T = x.shape
        H = self.hidden_dim
        vl = _lengths_tensor(lengths, B, T, x.device)
        if vl is not None:
            mask = _frame_mask(vl, T)
        m2 = _mask2d(mask)
        lens = None if m2 is None or vl is not None else m2.sum(dim=1).to(torch.int32)   # prefix masks (sequence_mask)
        # per item: the input's padding is masked out of the first operand, and the first GLU block's output too (its
        # own run's second GLU conv sees zero padding there)
        h = _conv(x, self._f_s0, mask=None if vl is None else m2)           # spectral.0
        h = _conv(h, self._f_s3, mode=ops.PACK_MISH)                        # mish -> spectral.3
        ops.frame_op(ops.OP_MISH, h, None, None, m2, h, None, B, H, T)      # mish(...) * mask
        h = self.temporal[0].run(h, None if vl is None else m2)
        h = self.temporal[1].run(h, m2)                                     # temporal(x) * mask
        y = self.slf_attn.run(h, lens, vl)
        ops.frame_op(ops.OP_ADD, h, y, None, None, h, None, B, H, T)
        h = _conv(h, self._f_fc)
        return ops.masked_mean(h, m2, **_vl(vl))


# ----------------------------------------------------------------------------------------------
# the inference paths of SynthesizerTrn  (hierspeechpp_speechsynthesizer.py:562-699)
# ----------------------------------------------------------------------------------------------
def sequence_mask(length, max_length=None):
    """commons.py:128-132."""
    if max_length is None:
        max_length = length.max()
    x = torch.arange(max_length, dtype=length.dtype, device=length.device)
    return x.unsqueeze(0) < length.unsqueeze(1)


class HierSpeechSynthesizer(nn.Module):
    """The modules ``SynthesizerTrn.infer`` / ``voice_conversion`` / ``voice_conversion_noise_control`` use, under the
    reference's attribute names (``enc_p_l, flow_l, flow, sn, dec, emb_g``), so ``load_state_dict(ckpt, strict=False)``
    takes a reference checkpoint (its training-only ``enc_p / enc_q / mel_decoder`` entries are reported as unexpected)."""

    def __init__(self, inter_channels=192, hidden_channels=192, resblock_kernel_sizes=(3, 7, 11),
                 resblock_dilation_sizes=((1, 3, 5), (1, 3, 5), (1, 3, 5)), upsample_rates=(4, 5, 4, 2, 2),
                 upsample_initial_channel=512, upsample_kernel_sizes=(8, 11, 8, 4, 4), gin_channels=256, **kwargs):
        super().__init__()
        self.enc_p_l = PosteriorSFEncoder(1024, inter_channels, hidden_channels, 5, 1, 16, gin_channels=gin_channels)
        self.flow_l = ResidualCouplingBlock_Transformer(inter_channels, hidden_channels, 5, 1, 3, gin_channels=gin_channels)
        self.flow = ResidualCouplingBlock_Transformer(inter_channels, hidden_channels, 5, 1, 3, gin_channels=gin_channels)
        self.dec = Generator(inter_channels, list(resblock_kernel_sizes), [list(d) for d in resblock_dilation_sizes],
                             list(upsample_rates), upsample_initial_channel, list(upsample_kernel_sizes),
                             gin_channels=gin_channels)
        self.sn = SourceNetwork(upsample_initial_channel // 2)
        self.emb_g = StyleEncoder(in_dim=80, hidden_dim=256, out_dim=gin_channels)

    @torch.no_grad()
    def infer(self, x_mel, w2v, length, f0, *, per_item=False, eps=None, seed=None):
        """``per_item``: see ``voice_conversion_noise_control``; x_mel [B, 80, T] shares ``length`` with w2v, and ``eps`` /
        ``seed`` give the draw inside ``enc_p_l`` (:201).  Returns (waveform, pitch prediction) as the reference does."""
        if per_item:
            vl, _, seeds = self._per_item_args(w2v, length, f0, x_mel, None, w2v.shape[0], eps, seed)
            g = self.emb_g(_as_input(x_mel), lengths=vl).unsqueeze(-1)
            return self._convert(w2v, vl, f0, g, eps, 1.0, need_pred=True, seeds=seeds)
        _no_eps(eps)
        _per_item_noise_args(False, 0, None, None, seed)
        x_mask = torch.unsqueeze(sequence_mask(length, x_mel.size(2)), 1).to(x_mel.dtype)
        g = self.emb_g(x_mel, x_mask).unsqueeze(-1)
        z, _, _ = self.enc_p_l(w2v, f0, x_mask, g=g)
        z = self.flow_l(z, x_mask, g=g, reverse=True)
        z = self.flow(z, x_mask, g=g, reverse=True)
        return vocode(self.sn, self.dec, z, g, need_pred=True)

    @torch.no_grad()
    def voice_conversion_noise_control(self, src, src_length, trg_mel, trg_length, f0, noise_scale=0.333, uncond=False,
                                       denoise_ratio=0, *, per_item=False, eps=None, seed=None):
        """``per_item=True``: B utterances of different lengths padded into one batch, each computed exactly as this
        method (``per_item=False``) computes it alone -- batch 1, unpadded, its own prompts, the same noise -- bit for bit.

        * ``src`` [B, 1024, T] padded; ``src_length`` = frames per item: an int CUDA tensor [B] (never read back, so the
          call stays capturable) or a host sequence (range-checked to [1, T]).  ``f0`` [B, 1, 4T].
        * ``trg_mel`` [2B, 80, Tm]: rows [0, B) are each item's prompt, rows [B, 2B) its denoised prompt (B = 1 is the
          reference's [2, 80, Tm] layout); ``trg_length`` [2B].  Item b uses (1 - r) g[b] + r g[B + b].  (Equality with
          the item's own call holds when its two prompts have the same length: the own call pads them to each other.)
        * ``eps``: fp32 CUDA [B, 192, T], the noise multiplying exp(logs_p) (the reference's second draw, :687); item b
          uses eps[b, :, :len[b]].  With ``eps=None`` and ``seed=None`` one ``randn`` of the padded shape is drawn:
          capturable, but then an item's noise depends on the batch it is in.
        * ``seed`` (instead of ``eps``): int64 CUDA tensor [B] or host sequence of 64-bit seeds.  Item b's noise is
          generated from seed[b] on the device, inside the sampling launch, and equals
          ``eps = ops.seeded_normal(seed[b:b+1], 192, len[b])`` of its own call: same request, same seed, same audio, in
          any batch.  This is the project's own generator (Philox4x32-10), not torch's ``randn`` stream.
        * ``noise_scale`` and ``denoise_ratio`` may be floating CUDA tensors [B], one value per item: item b equals its
          own call with ``float(noise_scale[b])`` and ``float(denoise_ratio[b])`` (noise_scale rounded to fp32 once,
          1 - r evaluated in float64 and then rounded, as the Python-float call does).  As device tensors they are
          inputs of a captured graph, so one graph serves every mix of seeds and controls.
        * Nothing past an item's length is read (any finite padding gives the same result); the waveform is
          [B, 1, 320 T] with item b's samples past 320 len[b] exactly 0."""
        if uncond:
            raise NotImplementedError("classifier-free guidance branch (cfg=True models) is not on this path")
        if per_item:
            B = src.shape[0]
            vl, tl, seeds = self._per_item_args(src, src_length, f0, trg_mel, trg_length, 2 * B, eps, seed,
                                                noise_scale=noise_scale, denoise_ratio=denoise_ratio)
            g = self.emb_g(_as_input(trg_mel), lengths=tl).unsqueeze(-1)
            if _per_item_control(denoise_ratio, B, src.device):
                # the scalar call's arithmetic per item: (1 - r) in float64, both weights rounded to fp32, fp32 products
                r = denoise_ratio.detach().to(torch.float64).view(B, 1, 1)
                g = ((1 - r).float() * g[:B] + r.float() * g[B:]).contiguous()
            else:
                g = ((1 - denoise_ratio) * g[:B] + denoise_ratio * g[B:]).contiguous()
            return self._convert(src, vl, f0, g, eps, noise_scale, seeds=seeds)[0]
        _no_eps(eps)
        _per_item_noise_args(False, 0, None, None, seed, noise_scale=noise_scale, denoise_ratio=denoise_ratio)
        trg_mask = torch.unsqueeze(sequence_mask(trg_length, trg_mel.size(2)), 1).to(trg_mel.dtype)
        g = self.emb_g(trg_mel, trg_mask).unsqueeze(-1)
        g_org, g_denoise = g[:1, :, :], g[1:, :, :]
        g_interpolation = ((1 - denoise_ratio) * g_org + denoise_ratio * g_denoise).contiguous()
        y_mask = torch.unsqueeze(sequence_mask(src_length, src.size(2)), 1).to(trg_mel.dtype)
        z, m_p, logs_p = self.enc_p_l(src, f0, y_mask, g=g_interpolation)
        B, C, T = m_p.shape
        eps = torch.randn_like(m_p)                                     # the second draw (:687)
        stats = torch.cat([m_p, logs_p], 1)
        ops.frame_op(ops.OP_SAMPLE, stats, eps.contiguous(), None, _mask2d(y_mask), z, None, B, C, T, s=float(noise_scale))
        z = self.flow_l(z, y_mask, g=g_interpolation, reverse=True)
        z = self.flow(z, y_mask, g=g_interpolation, reverse=True)
        return vocode(self.sn, self.dec, z, g_interpolation)[0]

    @torch.no_grad()
    def voice_conversion(self, src, src_length, trg_mel, trg_length, f0, noise_scale=0.333, uncond=False, *,
                         per_item=False, eps=None, seed=None):
        """``per_item``: see ``voice_conversion_noise_control``, with one prompt per item: ``trg_mel`` [B, 80, Tm]."""
        if uncond:
            raise NotImplementedError("classifier-free guidance branch (cfg=True models) is not on this path")
        if per_item:
            vl, tl, seeds = self._per_item_args(src, src_length, f0, trg_mel, trg_length, src.shape[0], eps, seed,
                                                noise_scale=noise_scale)
            g = self.emb_g(_as_input(trg_mel), lengths=tl).unsqueeze(-1)
            return self._convert(src, vl, f0, g, eps, noise_scale, seeds=seeds)[0]
        _no_eps(eps)
        _per_item_noise_args(False, 0, None, None, seed, noise_scale=noise_scale)
        trg_mask = torch.unsqueeze(sequence_mask(trg_length, trg_mel.size(2)), 1).to(trg_mel.dtype)
        g = self.emb_g(trg_mel, trg_mask).unsqueeze(-1)
        y_mask = torch.unsqueeze(sequence_mask(src_length, src.size(2)), 1).to(trg_mel.dtype)
        z, m_p, logs_p = self.enc_p_l(src, f0, y_mask, g=g)
        B, C, T = m_p.shape
        eps = torch.randn_like(m_p)
        stats = torch.cat([m_p, logs_p], 1)
        ops.frame_op(ops.OP_SAMPLE, stats, eps.contiguous(), None, _mask2d(y_mask), z, None, B, C, T, s=float(noise_scale))
        z = self.flow_l(z, y_mask, g=g, reverse=True)
        z = self.flow(z, y_mask, g=g, reverse=True)
        return vocode(self.sn, self.dec, z, g)[0]

    # ---- per-item batches
    def _per_item_args(self, src, src_length, f0, mel, mel_length, rows: int, eps, seed, **controls):
        """Checks every argument of a per-item call before anything runs; returns the int32 lengths of the source and
        of the prompts (``mel_length=None``: the prompts share the source's lengths and T, as ``infer``'s x_mel) and the
        int64 seeds (or None)."""
        if src.dim() != 3:
            raise ValueError(f"the source must be [B, C, T], got {tuple(src.shape)}")
        B, _, T = src.shape
        vl = _lengths_tensor(src_length, B, T, src.device)
        Tm = T if mel_length is None else (mel.shape[-1] if mel.dim() == 3 else -1)
        if tuple(mel.shape) != (rows, self.emb_g.in_dim, Tm):
            want = f"[{rows}, {self.emb_g.in_dim}, {'T' if mel_length is None else 'Tm'}]"
            raise ValueError(f"the prompt mel must be {want}, got {tuple(mel.shape)}")
        tl = vl if mel_length is None else _lengths_tensor(mel_length, rows, Tm, src.device)
        if tuple(f0.shape) != (B, 1, 4 * T):
            raise ValueError(f"f0 must be [{B}, 1, {4 * T}], got {tuple(f0.shape)}")
        if eps is not None:
            _check_eps(eps, B, self.enc_p_l.out_channels, T, src.device)
        seeds = _per_item_noise_args(True, B, src.device, eps, seed, **controls)
        return vl, tl, seeds

    def _convert(self, src, src_length, f0, g, eps, noise_scale, need_pred: bool = False, seeds=None):
        """enc_p_l -> flow_l -> flow -> vocoder of a per-item batch (g [B, gin, 1] per item); returns vocode's pair."""
        src, f0 = _as_input(src), _as_input(f0)
        B, _, T = src.shape
        vl = _lengths_tensor(src_length, B, T, src.device)
        if eps is None and seeds is None:
            eps = torch.randn(B, self.enc_p_l.out_channels, T, dtype=torch.float32, device=src.device)
        z, _, _ = self.enc_p_l(src, f0, None, g=g, eps=eps, noise_scale=noise_scale, lengths=vl, seed=seeds)
        z = self.flow_l(z, None, g=g, reverse=True, lengths=vl)
        z = self.flow(z, None, g=g, reverse=True, lengths=vl)
        return vocode(self.sn, self.dec, z, g, need_pred, lengths=vl)


def _no_eps(eps):
    if eps is not None:
        raise ValueError("eps= is taken with per_item=True (per_item=False draws the reference's noise itself)")
