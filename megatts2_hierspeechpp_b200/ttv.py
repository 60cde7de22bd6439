"""The tail of the text-to-vec model (SURVEY.md §8f4, partial), B200-native: ``W2VDecoder``
(ttv_v1/t2w2v_transformer.py:377-405) and ``PitchPredictor`` (:408-463; ``ResBlock1`` of ttv_v1/modules.py:187-223).

Both ``SynthesizerTrn.infer`` (:1109-1110) and ``inf_plm_gen`` (:991-992) end with
``w2v = w2v_decoder(z, y_mask, g); pitch = pp(w2v, g)`` and hand ``(w2v, pitch)`` to
``net_g.voice_conversion_noise_control`` (inference.py:158-167), i.e. to ``front.HierSpeechSynthesizer``: with these two
modules the device-resident chain starts at the flow output of the text-to-vec model.  The language-model sampling loop
and the text encoder before it are out of scope (DESIGN.md §7).

Same class names, constructor / forward signatures and ``state_dict`` keys as the reference.  Every Conv1d /
ConvTranspose1d runs on the tcgen05 conv kernel with leaky_relu fused into the operand pack; the 1/3 of the resblock
mean is folded into the consumer's pack (leaky_relu is positively homogeneous).  Inference only, CUDA tensors only."""
from __future__ import annotations

from typing import Optional, Sequence

import torch
from torch import nn
from torch.nn import Conv1d, ConvTranspose1d

from . import ops
from .front import WN, _conv, _mask2d, _vec
from .modules import (_Folded, _MAIN_SLOT, _as_input, _bump_on_load, _frame_mask, _hops, _length_table,
                      _lengths_tensor, _row_tiles, _vl, _weight_norm, get_padding, sum_of_blocks)

LRELU_SLOPE = 0.1
_SLOT2 = 12       # second operand workspace of a resblock stream (slots 0..2 -> 12..14)


class W2VDecoder(nn.Module):
    def __init__(self, in_channels, hidden_channels, kernel_size, dilation_rate, n_layers, output_size=1024,
                 gin_channels=0, p_dropout=0):
        super().__init__()
        self.in_channels = in_channels
        self.hidden_channels = hidden_channels
        self.kernel_size = kernel_size
        self.dilation_rate = dilation_rate
        self.n_layers = n_layers
        self.gin_channels = gin_channels
        self.p_dropout = p_dropout
        self.output_size = output_size
        self.pre = nn.Conv1d(in_channels, hidden_channels, 1)
        self.enc = WN(hidden_channels, kernel_size, dilation_rate, n_layers, gin_channels=gin_channels,
                      p_dropout=p_dropout)
        self.proj = nn.Conv1d(hidden_channels, output_size, 1)
        self._f_pre = _Folded(self.pre)
        self._f_proj = _Folded(self.proj)
        _bump_on_load(self)

    def forward(self, x, x_mask, g=None, *, lengths=None):
        """``lengths`` (frames per item: int CUDA tensor [B] or host sequence): a padded batch whose item b equals, bit for
        bit, its own unpadded run with ``x_mask`` = ones, with 0 past its length; ``x_mask`` is then derived from them (the
        one passed is not read) and x past an item is never used."""
        B, _, T = x.shape
        vl = _lengths_tensor(lengths, B, T, x.device)
        x = _as_input(x)
        if vl is not None:
            x_mask = _frame_mask(vl, T).unsqueeze(1)
        mask = _mask2d(x_mask)
        h = _conv(x, self._f_pre, mask=mask)                     # pre(x * x_mask)
        ops.frame_op(ops.OP_MASK, h, None, None, mask, h, None, B, self.hidden_channels, T)
        h = self.enc(h, x_mask, g=g)
        y = _conv(h, self._f_proj)
        ops.frame_op(ops.OP_MASK, y, None, None, mask, y, None, B, self.output_size, T)
        return y


class ResBlock1(nn.Module):
    """ttv_v1/modules.py:187-229 (``x_mask=None`` call of PitchPredictor)."""

    def __init__(self, channels, kernel_size=3, dilation=(1, 3, 5)):
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
        self._f1 = [_Folded(c) for c in self.convs1]
        self._f2 = [_Folded(c) for c in self.convs2]
        _bump_on_load(self)

    def run(self, x: torch.Tensor, slot: int = 0, acc: Optional[torch.Tensor] = None, acc_mode: int = ops.ACC_NONE,
            before_final=None, valid_len: Optional[torch.Tensor] = None) -> Optional[torch.Tensor]:
        """Same contract as ``AMPBlock1.run``: x is not modified; with ``acc`` the result is only accumulated.
        ``valid_len`` (int32 [B]): item b is x[b, :, :valid_len[b]]; the output below that equals the item's own run, past
        it it is not meaningful (every operand built from it is zero there, as in the item's own run)."""
        B, C, L = x.shape
        if C != self.channels or C % 16:
            raise ValueError(f"ResBlock1 expects {self.channels} channels (multiple of 16), got {C}")
        k = self.kernel_size
        buf = ops.blk16_buffer(B, C, L, x.device, slot)
        buf2 = ops.blk16_buffer(B, C, L, x.device, slot + _SLOT2)
        cur = x
        nl = len(self.dilation)
        rt = _row_tiles(B, L)
        mask = None if valid_len is None else _frame_mask(valid_len, L)
        for i, d in enumerate(self.dilation):
            last = i == nl - 1
            w1, nt1 = self._f1[i].packed_weight(rt)
            w2, nt2 = self._f2[i].packed_weight(rt)
            ops.pack_blk16(cur, buf, True, **_vl(valid_len))
            ops.check_saturation(buf, C, L)
            # c1's epilogue applies the second leaky_relu and writes c2's fp16 operand (no fp32 round trip, no pack);
            # with lengths, the mask gives that operand the zero tail of the item's own run
            ops.conv1d_umma_blk(buf, w1, self._f1[i].bias(), L, C, C, k, d, nt1, buf2, ops.BLK_LRELU, mask=mask)
            ops.check_saturation(buf2, C, L)
            buf, buf2 = buf2, buf
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

    def forward(self, x, x_mask=None):
        if x_mask is not None:
            raise NotImplementedError("ResBlock1: the masked variant is not on the inference path (PitchPredictor :449)")
        return self.run(_as_input(x))

    def remove_weight_norm(self):
        for l in list(self.convs1) + list(self.convs2):
            torch.nn.utils.remove_weight_norm(l)
        self._f1 = [_Folded(c) for c in self.convs1]
        self._f2 = [_Folded(c) for c in self.convs2]


class PitchPredictor(nn.Module):
    """[B,1024,T] w2v features + style vector -> [B,1,4T] log-f0 (ttv_v1/t2w2v_transformer.py:408-463)."""

    parallel_blocks = True     # one stream per resblock (they are 1-wave kernels)

    def __init__(self):
        super().__init__()
        resblock_kernel_sizes = [3, 5, 7]
        upsample_rates = [2, 2]
        initial_channel = 1024
        upsample_initial_channel = 256
        upsample_kernel_sizes = [4, 4]
        resblock_dilation_sizes = [[1, 3, 5], [1, 3, 5], [1, 3, 5]]
        self.num_kernels = len(resblock_kernel_sizes)
        self.num_upsamples = len(upsample_rates)
        self.upsample_rates = upsample_rates
        self.conv_pre = Conv1d(initial_channel, upsample_initial_channel, 7, 1, padding=3)
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
                self.resblocks.append(ResBlock1(ch, k, d))
        self.conv_post = Conv1d(ch, 1, 7, 1, padding=3, bias=False)
        self.cond = Conv1d(256, upsample_initial_channel, 1)
        self.softplus = torch.nn.Softplus()      # unused by forward, kept for the module tree of the reference
        self._f_pre = _Folded(self.conv_pre)
        self._f_ups = [_Folded(u) for u in self.ups]
        self._f_cond = _Folded(self.cond)
        self._f_post = _Folded(self.conv_post)
        self._post_key, self._post_w = None, None
        _bump_on_load(self)

    def _post_weight(self, scale: float) -> torch.Tensor:
        """conv_post weight times the pending 1/num_kernels: conv_post has no bias and leaky_relu(s*x) = s*leaky_relu(x)
        for s > 0, so the division of :454 moves onto the 448 weights."""
        w = self._f_post.weight()
        key = (self._f_post.key, scale)
        if key != self._post_key:
            self._post_w = (w * scale).contiguous()
            self._post_key = key
        return self._post_w

    def forward(self, x, g, *, lengths=None):
        """``lengths`` (frames of x per item: int CUDA tensor [B] or host sequence): a padded batch whose item b's pitch
        [:4 * lengths[b]] equals, bit for bit, its own unpadded run, with 0 past it; x past an item is never used.
        ``lengths=None`` is the reference's call, which runs the padding through like any other frame."""
        B, _, T = x.shape
        V = _length_table(lengths, B, T, x.device, _hops(self.upsample_rates))
        vl = (lambda i: None) if V is None else (lambda i: V[i])
        x, g = _as_input(x), _as_input(g)
        c0 = self.conv_pre.out_channels
        if V is None:
            h = _conv(x, self._f_pre, k=7)                                    # split-K over the 1024 input channels
        else:   # the batch-1 split-K launches at every B; padding never enters the operand
            h = _conv(x, self._f_pre, k=7, mask=_frame_mask(V[0], T), strided=True)
        cg = _vec(g.reshape(B, -1), self._f_cond)
        ops.frame_op(ops.OP_ADD_BCAST, h, None, cg, None, h, None, B, c0, T, cstride=c0)
        sc = 1.0
        L = T
        for i in range(self.num_upsamples):
            cin = (h[0] if isinstance(h, list) else h).shape[1]
            f = self._f_ups[i]
            buf = ops.blk16_buffer(B, cin, L, x.device, _MAIN_SLOT)
            ops.pack_blk16(h, buf, True, scale=sc, **_vl(vl(i)))             # leaky_relu(x / num_kernels, 0.1)
            ops.check_saturation(buf, cin, L)
            wp, nt = f.packedT_weight(self.upsample_rates[i], _row_tiles(B, L))
            h = ops.conv_transpose1d_umma(buf, wp, f.bias(), L, cin, f.conv.out_channels,
                                          self.ups[i].kernel_size[0], self.upsample_rates[i], nt)
            L *= self.upsample_rates[i]
            blocks: Sequence[ResBlock1] = self.resblocks[i * self.num_kernels:(i + 1) * self.num_kernels]
            h, sc = sum_of_blocks(h, blocks, parallel=self.parallel_blocks, separate=i < self.num_upsamples - 1,
                                  valid_len=vl(i + 1))
        return ops.conv1d_direct(h, self._post_weight(sc), None, pad=3, flags=ops.CONV_LRELU001_IN,
                                 **_vl(vl(self.num_upsamples)))

    def remove_weight_norm(self):
        for l in self.ups:
            torch.nn.utils.remove_weight_norm(l)
        for l in self.resblocks:
            l.remove_weight_norm()
        self._f_ups = [_Folded(u) for u in self.ups]


class TTVTail(nn.Module):
    """``w2v_decoder`` + ``pp`` under the reference's attribute names, so a text-to-vec checkpoint's
    ``w2v_decoder.*`` / ``pp.*`` entries load with ``load_state_dict(..., strict=False)`` and the synthetic
    ``ttv_tail_sd`` loads strictly.  ``forward(z, y_mask, g) -> (w2v, pitch)`` (:1109-1110).

    ``forward(z, y_mask, g, lengths=...)`` (frames of z per item: int CUDA tensor [B] or host sequence): a padded batch
    whose item b's w2v [:lengths[b]] and pitch [:4 * lengths[b]] equal, bit for bit, ``forward`` on that item alone with
    ``y_mask`` = ones, with 0 past them; ``y_mask`` may be passed but is not read, and z past an item is never used.
    Its outputs go on as they are to ``HierSpeechSynthesizer.voice_conversion_noise_control(w2v, lengths, ..., pitch,
    per_item=True)``."""

    def __init__(self, inter_channels: int = 256, gin_channels: int = 256):
        super().__init__()
        self.w2v_decoder = W2VDecoder(inter_channels, inter_channels * 2, 5, 1, 8, output_size=1024, p_dropout=0.1,
                                      gin_channels=gin_channels)
        self.pp = PitchPredictor()

    def forward(self, z, y_mask, g, *, lengths=None):
        vl = _lengths_tensor(lengths, z.shape[0], z.shape[-1], z.device)
        w2v = self.w2v_decoder(z, y_mask, g=g, lengths=vl)
        return w2v, self.pp(w2v, g, lengths=vl)
