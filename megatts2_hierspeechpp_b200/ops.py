"""Tensor-level wrappers over the hsv C-ABI (``include/hsv.h``).

PyTorch is used only for device memory and streams: every function here checks
its arguments, takes raw device pointers and launches a hand-written sm_100a
kernel on ``torch.cuda.current_stream()``.  No function has a CPU path.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional, Tuple

import torch

from . import _lib

BLK_PAD = 32
TILE_M = 128
BLK_ROUND = 512

CONV_LRELU_IN = 1
CONV_TANH = 2
CONV_ADD_OUT = 4

ACC_NONE, ACC_SET, ACC_ADD = 0, 1, 2


def _p(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _req(t: torch.Tensor, name: str, dtype=torch.float32, ndim: Optional[int] = None):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name}: expected a CUDA tensor (no CPU fallback), got device {t.device}")
    if t.dtype != dtype:
        raise ValueError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name}: expected a contiguous tensor")
    if ndim is not None and t.dim() != ndim:
        raise ValueError(f"{name}: expected {ndim} dims, got shape {tuple(t.shape)}")


def blk16_rows(L: int) -> int:
    return 2 * BLK_PAD + ((L + BLK_ROUND - 1) // BLK_ROUND) * BLK_ROUND


def blk_cw(C: int) -> int:
    """Channels per operand row of the swizzled blk16 layout (include/hsv.h)."""
    return 64 if C % 64 == 0 else (32 if C % 32 == 0 else 16)


def blk16_shape(B: int, C: int, L: int) -> Tuple[int, int, int, int]:
    if C % 16:
        raise ValueError(f"blk16 needs C % 16 == 0 (C={C})")
    cw = blk_cw(C)
    return (B, C // cw, blk16_rows(L), cw)


# Operand workspaces are cached per exact (device, B, C, L, slot) -- the layout's zero rows around the sequence
# must survive reuse, so a buffer is only ever reused for the shape it was zero-initialised for.  The cache is an
# LRU bounded in bytes (WORKSPACE_BUDGET_BYTES; variable-length serving would otherwise grow it without bound).
# Evicting or clearing bumps WORKSPACE_EPOCH, which invalidates every captured CUDA graph that baked the old
# pointers in (runtime.CudaGraphRunner keys on it).
from collections import OrderedDict

_blk_pool: "OrderedDict[Tuple, torch.Tensor]" = OrderedDict()
WORKSPACE_BUDGET_BYTES = [int(__import__("os").environ.get("HSV_WORKSPACE_BUDGET_MB", "16384")) << 20]
WORKSPACE_EPOCH = [0]
_pin_depth = [0]      # > 0 while a CUDA graph is being warmed up / captured: no eviction in that window


def workspace_bytes() -> int:
    return sum(b.numel() * b.element_size() for b in _blk_pool.values())


def blk16_buffer(B: int, C: int, L: int, device, slot: int = 0) -> torch.Tensor:
    """Zero-initialised fp16 [B, C/CW, Lp, CW] operand buffer (opaque, swizzled), cached per shape.

    Producers only ever write rows [BLK_PAD, BLK_PAD+L), so the zero rows that
    implement the conv's zero padding survive reuse."""
    dev = torch.device(device)
    key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device(), B, C, L, slot)
    buf = _blk_pool.get(key)
    if buf is not None:
        _blk_pool.move_to_end(key)
        return buf
    shape = blk16_shape(B, C, L)
    need = 2 * shape[0] * shape[1] * shape[2] * shape[3]
    if _pin_depth[0] == 0:
        evicted = False
        while _blk_pool and workspace_bytes() + need > WORKSPACE_BUDGET_BYTES[0]:
            _blk_pool.popitem(last=False)
            evicted = True
        if evicted:
            WORKSPACE_EPOCH[0] += 1
    buf = torch.zeros(*shape, dtype=torch.float16, device=dev)
    _blk_pool[key] = buf
    return buf


def clear_workspace():
    _blk_pool.clear()
    WORKSPACE_EPOCH[0] += 1


def _req_len(valid_len: Optional[torch.Tensor], B: int, device, name: str = "valid_len"):
    """Per-item valid lengths of a ragged batch: a contiguous int32 CUDA tensor [B] on the data's device (values are
    clamped to [0, L] by the kernels)."""
    if valid_len is None:
        return
    _req(valid_len, name, torch.int32, 1)
    if valid_len.numel() != B:
        raise ValueError(f"{name}: expected {B} elements, got {valid_len.numel()}")
    if valid_len.device != torch.device(device):
        raise ValueError(f"{name}: on {valid_len.device}, the data is on {device}")


def act1d(x: torch.Tensor, alpha: torch.Tensor, beta: torch.Tensor, out: Optional[torch.Tensor] = None,
          scale: float = 1.0, valid_len: Optional[torch.Tensor] = None):
    """Fused Activation1d(SnakeBeta) of ``x * scale``: fp32 [B,C,L] -> fp32 [B,C,L].  ``valid_len`` (int32 [B]): item b
    is its first valid_len[b] steps, as if run alone; the rest of its output is 0 and the rest of its input unread."""
    _req(x, "x", ndim=3); _req(alpha, "alpha"); _req(beta, "beta")
    B, C, L = x.shape
    if alpha.numel() != C or beta.numel() != C:
        raise ValueError(f"alpha/beta must have {C} elements")
    _req_len(valid_len, B, x.device)
    if out is None:
        out = torch.empty_like(x)
    else:
        _req(out, "out", ndim=3)
    lib = _lib.load()
    _lib.check(lib.hsv_act1d_snakebeta_ragged(_p(x), _p(out), _p(alpha), _p(beta), _p(valid_len), B, C, L, 0,
                                              float(scale), _stream()), "hsv_act1d_snakebeta")
    return out


def act1d_blk16(x: torch.Tensor, alpha: torch.Tensor, beta: torch.Tensor, buf: torch.Tensor, scale: float = 1.0,
                valid_len: Optional[torch.Tensor] = None):
    """Fused Activation1d(SnakeBeta) of ``x * scale``: fp32 [B,C,L] -> fp16 blk16 operand (into ``buf``).
    ``valid_len``: as ``act1d`` (operand rows past an item's length are written as zero)."""
    _req(x, "x", ndim=3); _req(alpha, "alpha"); _req(beta, "beta"); _req(buf, "buf", torch.float16, 4)
    B, C, L = x.shape
    if tuple(buf.shape) != blk16_shape(B, C, L):
        raise ValueError(f"blk16 buffer shape {tuple(buf.shape)} does not match x {tuple(x.shape)}")
    _req_len(valid_len, B, x.device)
    lib = _lib.load()
    _lib.check(lib.hsv_act1d_snakebeta_ragged(_p(x), _p(buf), _p(alpha), _p(beta), _p(valid_len), B, C, L, 1,
                                              float(scale), _stream()), "hsv_act1d_snakebeta")
    return buf


def pack_blk16(x, buf: torch.Tensor, lrelu: bool = False, scale: float = 1.0, valid_len: Optional[torch.Tensor] = None):
    """fp32 [B,C,L] -> fp16 blk16 operand of ``x * scale`` (optionally leaky_relu(0.1) of it).  ``x`` may be a list of up
    to three equally shaped tensors: the operand is then ``((x1 + x2) + x3) * scale`` (the sum over a stage's resblocks
    taken by the consumer, ``modules.sum_of_blocks(..., separate=True)``).  ``valid_len`` (int32 [B]): operand rows at
    t >= valid_len[b] are written as zero without reading x."""
    xs = list(x) if isinstance(x, (list, tuple)) else [x]
    if not 1 <= len(xs) <= 3:
        raise ValueError("pack_blk16: one to three addends")
    for t in xs:
        _req(t, "x", ndim=3)
        if t.shape != xs[0].shape:
            raise ValueError("pack_blk16: addend shapes differ")
    _req(buf, "buf", torch.float16, 4)
    B, C, L = xs[0].shape
    if tuple(buf.shape) != blk16_shape(B, C, L):
        raise ValueError("blk16 buffer shape mismatch")
    lib = _lib.load()
    if valid_len is not None:
        _req_len(valid_len, B, xs[0].device)
        xs = xs + [None] * (3 - len(xs))
        _lib.check(lib.hsv_pack_blk16_sum3_ragged(_p(xs[0]), _p(xs[1]), _p(xs[2]), _p(valid_len), _p(buf), B, C, L,
                                                  int(lrelu), float(scale), _stream()), "hsv_pack_blk16_sum3_ragged")
    elif len(xs) == 1:
        _lib.check(lib.hsv_pack_blk16(_p(xs[0]), _p(buf), B, C, L, int(lrelu), float(scale), _stream()), "hsv_pack_blk16")
    else:
        _lib.check(lib.hsv_pack_blk16_sum3(_p(xs[0]), _p(xs[1]), _p(xs[2]) if len(xs) == 3 else None, _p(buf), B, C, L,
                                           int(lrelu), float(scale), _stream()), "hsv_pack_blk16_sum3")
    return buf


def unpack_blk16(buf: torch.Tensor, C: int, L: int) -> torch.Tensor:
    """fp16 blk16 operand buffer -> fp32 [B,C,L] (tests / debugging)."""
    _req(buf, "buf", torch.float16, 4)
    B = buf.shape[0]
    if tuple(buf.shape) != blk16_shape(B, C, L):
        raise ValueError("blk16 buffer shape mismatch")
    out = torch.empty(B, C, L, dtype=torch.float32, device=buf.device)
    lib = _lib.load()
    _lib.check(lib.hsv_unpack_blk16(_p(buf), _p(out), B, C, L, _stream()), "hsv_unpack_blk16")
    return out


def blk16_stats(buf: torch.Tensor, C: int, L: int, stats: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Operand health of a blk16 buffer: int32 [2] = (count of non-finite fp16 values, float bits of max |value|),
    accumulated into ``stats`` (zeroed by the caller) or a fresh tensor.  Debugging aid: the reference keeps fp32
    activations, the tensor-core operands here are fp16 and saturate beyond +-65504."""
    _req(buf, "buf", torch.float16, 4)
    B = buf.shape[0]
    if tuple(buf.shape) != blk16_shape(B, C, L):
        raise ValueError("blk16 buffer shape mismatch")
    if stats is None:
        stats = torch.zeros(2, dtype=torch.int32, device=buf.device)
    lib = _lib.load()
    _lib.check(lib.hsv_blk16_stats(_p(buf), _p(stats), B, C, L, _stream()), "hsv_blk16_stats")
    return stats


SATURATION = {"enabled": bool(int(__import__("os").environ.get("HSV_CHECK_SATURATION", "0"))), "stats": None}


def check_saturation(buf: torch.Tensor, C: int, L: int):
    """Called by the module layer after every operand producer when HSV_CHECK_SATURATION=1 (or
    ``ops.SATURATION["enabled"] = True``): accumulates into one device counter, no host sync;
    ``saturation_report()`` reads it."""
    if not SATURATION["enabled"]:
        return
    if SATURATION["stats"] is None or SATURATION["stats"].device != buf.device:
        SATURATION["stats"] = torch.zeros(2, dtype=torch.int32, device=buf.device)
    blk16_stats(buf, C, L, SATURATION["stats"])


def saturation_report(reset: bool = True):
    """(non-finite operand values seen, largest finite |operand|) since the last reset; raises nothing."""
    st = SATURATION["stats"]
    if st is None:
        return 0, 0.0
    n, mx = int(st[0].item()), float(st[1:2].view(torch.float32).item())
    if reset:
        st.zero_()
    return n, mx


def _static_data_barrier(what: str):
    """The conv / activation kernels are launched with programmatic dependent launch and read their STATIC inputs
    (packed weights, bias, alpha/beta) BEFORE ``griddepcontrol.wait``, i.e. possibly while the kernel launched just
    before them on the stream is still running.  Kernels that PRODUCE static data (weight fold / pack: once per
    checkpoint and n_tile) therefore end with a stream synchronisation, so that nothing launched later can overlap
    them.  They cannot run inside a CUDA-graph capture (warm up once before capturing: CudaGraphRunner does)."""
    if torch.cuda.is_current_stream_capturing():
        raise RuntimeError(f"{what}: weights are being folded / packed inside a CUDA-graph capture; run one eager "
                           "forward first (weights are static data of the PDL-launched kernels)")
    torch.cuda.current_stream().synchronize()


def weight_norm_fold(v: torch.Tensor, g: torch.Tensor) -> torch.Tensor:
    """w = v * g/||v|| (norm over all dims but 0) == torch._weight_norm(v, g, 0)."""
    _req(v, "weight_v"); _req(g, "weight_g")
    n0 = v.shape[0]
    if g.numel() != n0:
        raise ValueError("weight_g must have one element per dim-0 slice of weight_v")
    w = torch.empty_like(v)
    lib = _lib.load()
    _lib.check(lib.hsv_weight_norm_fold(_p(v), _p(g), _p(w), n0, v.numel() // n0, _stream()), "hsv_weight_norm_fold")
    _static_data_barrier("weight_norm_fold")
    return w


def pick_n_tile(cout: int, row_tiles: int = 1 << 30, cin_taps: int = 1 << 30) -> int:
    """Output-channel tile of the tcgen05 conv (measured policy, tools/microbench4.py).  ``row_tiles`` = number of
    128-row tiles x batch x phases of the launch: with few row tiles (batch-1 latency regime) a narrower n_tile
    puts more CTAs to work on the same layer (shorter serial MMA chain and weight stream per CTA); with many, a
    wide tile has the best tensor/shared-memory efficiency -- 128, not 256 (746 vs 725 TFLOP/s at C = 256), and
    64 for the HBM-bound light layers (``cin_taps`` = Cin x taps < 512: 3.9 vs 3.4 TB/s at C = 128, k = 3)."""
    widest = (128, 64, 32, 16) if cin_taps >= 512 else (64, 32, 16)
    cands = [n for n in widest if cout % n == 0]
    if not cands:
        for n in range(widest[0], 15, -16):
            if cout % n == 0:
                cands = [n]
                break
    if not cands:
        raise ValueError(f"Cout={cout} not a multiple of 16")
    for n in cands:
        if n <= 32 or row_tiles * (cout // n) >= (120 if n >= 128 else 60):
            return n
    return cands[-1]


def pack_conv_weight(w: torch.Tensor, n_tile: int) -> torch.Tensor:
    _req(w, "w", ndim=3)
    cout, cin, k = w.shape
    out = torch.empty(cout * cin * k, dtype=torch.float16, device=w.device)
    lib = _lib.load()
    _lib.check(lib.hsv_pack_conv_weight(_p(w), _p(out), cout, cin, k, n_tile, _stream()), "hsv_pack_conv_weight")
    _static_data_barrier("pack_conv_weight")
    return out


def conv1d_umma(a_blk: torch.Tensor, w_packed: torch.Tensor, bias: Optional[torch.Tensor], L: int, cin: int,
                cout: int, k: int, d: int, n_tile: int, residual: Optional[torch.Tensor] = None,
                out: Optional[torch.Tensor] = None, acc: Optional[torch.Tensor] = None, acc_mode: int = ACC_NONE,
                acc_div: float = 1.0, want_out: bool = True):
    """tcgen05 implicit-GEMM Conv1d.  Returns ``out`` (fp32 [B,Cout,L]) or None if want_out=False.

    ``a_blk`` may also be a channel range of a wider blk16 buffer, ``buf[:, c0 // CW:(c0 + cin) // CW]`` with the same
    CW (a split-K pass over one packed operand): read in place through the A operand's batch stride."""
    _req_blk_view(a_blk, "a_blk16")
    _req(w_packed, "w_packed", torch.float16)
    B = a_blk.shape[0]
    if tuple(a_blk.shape) != blk16_shape(B, cin, L):
        raise ValueError(f"a_blk16 shape {tuple(a_blk.shape)} does not match Cin={cin}, L={L}")
    if w_packed.numel() < cout * cin * k:
        raise ValueError("w_packed size mismatch")
    for t, n in ((bias, "bias"), (residual, "residual"), (out, "out"), (acc, "acc")):
        if t is not None:
            _req(t, n)
    if residual is not None and tuple(residual.shape) != (B, cout, L):
        raise ValueError("residual shape mismatch")
    if out is None and want_out:
        out = torch.empty(B, cout, L, dtype=torch.float32, device=a_blk.device)
    if out is not None and tuple(out.shape) != (B, cout, L):
        raise ValueError("out shape mismatch")
    if acc is not None and tuple(acc.shape) != (B, cout, L):
        raise ValueError("acc shape mismatch")
    lib = _lib.load()
    if a_blk.is_contiguous():
        _lib.check(lib.hsv_conv1d_umma(_p(a_blk), _p(w_packed), _p(bias), _p(residual), _p(out), _p(acc), acc_mode,
                                       float(acc_div), B, cin, cout, L, k, d, n_tile, _stream()), "hsv_conv1d_umma")
    else:
        _lib.check(lib.hsv_conv1d_umma_astride(_p(a_blk), a_blk.stride(0) // a_blk.stride(1), _p(w_packed), _p(bias),
                                               _p(residual), _p(out), _p(acc), acc_mode, B, cin, cout, L, k, d, n_tile,
                                               _stream()), "hsv_conv1d_umma_astride")
    return out


def _req_blk_view(t: torch.Tensor, name: str):
    """A blk16 operand: a contiguous buffer, or a chunk range of one (dense inside each batch item, any batch stride)."""
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float16 and t.dim() == 4) or t.is_contiguous():
        _req(t, name, torch.float16, 4)
        return
    _, nc, rows, cw = t.shape
    if t.stride(3) != 1 or t.stride(2) != cw or t.stride(1) != rows * cw or t.stride(0) % t.stride(1):
        raise ValueError(f"{name}: a non-contiguous operand must be a chunk range of a contiguous blk16 buffer")


BLK_NONE, BLK_GATE, BLK_GELU, BLK_LRELU = 0, 1, 2, 3


def gate_permutation(two_h: int, device=None) -> torch.Tensor:
    """Output-channel order the operand-writing gate epilogue expects of a WN in_layer (2H channels: tanh half, sigmoid
    half): groups of [8 tanh | 8 sigmoid] = channels 8j..8j+7 then H+8j..H+8j+7."""
    H = two_h // 2
    if H % 8:
        raise ValueError("gate_permutation: H % 8 != 0")
    j = torch.arange(H // 8).view(-1, 1) * 8
    e = torch.arange(8).view(1, -1)
    return torch.cat([j + e, H + j + e], 1).reshape(-1).to(device)


def conv1d_umma_blk(a_blk: torch.Tensor, w_packed: torch.Tensor, bias: Optional[torch.Tensor], L: int, cin: int, cout: int,
                    k: int, d: int, n_tile: int, out_blk: torch.Tensor, mode: int = BLK_NONE,
                    bc: Optional[torch.Tensor] = None, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """tcgen05 Conv1d whose epilogue writes the NEXT conv's fp16 blk16 operand: act(conv + bias + bc[b]) * mask.
    ``bc``: [B, cout] rows (dense innermost dimension, any batch stride); BLK_GATE: weights / bias / bc in
    ``gate_permutation`` order, ``out_blk`` has cout // 2 channels."""
    _req(a_blk, "a_blk16", torch.float16, 4); _req(w_packed, "w_packed", torch.float16)
    _req(out_blk, "out_blk16", torch.float16, 4)
    B = a_blk.shape[0]
    if tuple(a_blk.shape) != blk16_shape(B, cin, L):
        raise ValueError(f"a_blk16 shape {tuple(a_blk.shape)} does not match Cin={cin}, L={L}")
    co = cout // 2 if mode == BLK_GATE else cout
    if tuple(out_blk.shape) != blk16_shape(B, co, L):
        raise ValueError(f"out_blk16 shape {tuple(out_blk.shape)} does not match C={co}, L={L}")
    if w_packed.numel() < cout * cin * k:
        raise ValueError("w_packed size mismatch")
    if bias is not None:
        _req(bias, "bias")
    bcs = 0
    if bc is not None:
        _req_vec(bc, "bc")
        if tuple(bc.shape) != (B, cout):
            raise ValueError("bc shape mismatch")
        bcs = bc.stride(0)
    if mask is not None:
        _req(mask, "mask")
    _lib.check(_lib.load().hsv_conv1d_umma_blk16(_p(a_blk), _p(w_packed), _p(bias), _p(out_blk), int(mode), _p(bc), int(bcs),
                                                 _p(mask), B, cin, cout, L, k, d, n_tile, _stream()),
               "hsv_conv1d_umma_blk16")
    return out_blk


def conv1d_umma_wn_tail(a_blk: torch.Tensor, w_packed: torch.Tensor, bias: Optional[torch.Tensor], x: torch.Tensor,
                        output: torch.Tensor, mask: Optional[torch.Tensor], next_blk: torch.Tensor, n_tile: int):
    """A WN layer's res_skip conv (1x1, Cin -> 2H) with the layer tail in its epilogue: x = (x + rs[:, :H]) * mask and
    output += rs[:, H:] in place, the new x also written as the next in_layer's fp16 operand ``next_blk``."""
    _req(a_blk, "a_blk16", torch.float16, 4); _req(w_packed, "w_packed", torch.float16)
    _req(next_blk, "next_blk16", torch.float16, 4); _req(x, "x", ndim=3); _req(output, "output", ndim=3)
    B, H, L = x.shape
    cin = a_blk.shape[1] * a_blk.shape[3]
    if tuple(a_blk.shape) != blk16_shape(B, cin, L) or tuple(next_blk.shape) != blk16_shape(B, H, L):
        raise ValueError("conv1d_umma_wn_tail: operand buffer shape mismatch")
    if tuple(output.shape) != (B, H, L) or H % n_tile:
        raise ValueError("conv1d_umma_wn_tail: output shape / n_tile mismatch")
    if bias is not None:
        _req(bias, "bias")
    if mask is not None:
        _req(mask, "mask")
    _lib.check(_lib.load().hsv_conv1d_umma_wn_tail(_p(a_blk), _p(w_packed), _p(bias), _p(x), _p(output), _p(mask),
                                                   _p(next_blk), B, cin, H, L, n_tile, _stream()), "hsv_conv1d_umma_wn_tail")
    return next_blk


def act_conv1d_umma(x: torch.Tensor, alpha: torch.Tensor, beta: torch.Tensor, w_packed: torch.Tensor,
                    bias: Optional[torch.Tensor], cout: int, k: int, d: int, residual: Optional[torch.Tensor] = None,
                    out: Optional[torch.Tensor] = None, acc: Optional[torch.Tensor] = None, acc_mode: int = ACC_NONE,
                    scale: float = 1.0, want_out: bool = True):
    """Whole AMP half-layer in one kernel: ``conv1d(Activation1d(x * scale))`` (+bias, +residual, accumulate).

    x fp32 [B,Cin,L] with Cin in {16,32,64}; ``w_packed`` from ``pack_conv_weight(w, n_tile=cout)``.  Bit-identical to
    ``act1d_blk16`` + ``conv1d_umma``; the fp16 operand never goes to HBM.  ``out``/``acc`` must not alias ``x``."""
    _req(x, "x", ndim=3); _req(alpha, "alpha"); _req(beta, "beta"); _req(w_packed, "w_packed", torch.float16)
    B, cin, L = x.shape
    if cin not in FUSED_CIN:
        raise ValueError(f"act_conv1d_umma: Cin must be one of {FUSED_CIN} (Cin={cin})")
    if alpha.numel() != cin or beta.numel() != cin:
        raise ValueError(f"alpha/beta must have {cin} elements")
    if w_packed.numel() < cout * cin * k:
        raise ValueError("w_packed size mismatch")
    for t, n in ((bias, "bias"), (residual, "residual"), (out, "out"), (acc, "acc")):
        if t is not None:
            _req(t, n)
    if residual is not None and tuple(residual.shape) != (B, cout, L):
        raise ValueError("residual shape mismatch")
    if out is None and want_out:
        out = torch.empty(B, cout, L, dtype=torch.float32, device=x.device)
    if out is not None and tuple(out.shape) != (B, cout, L):
        raise ValueError("out shape mismatch")
    if acc is not None and tuple(acc.shape) != (B, cout, L):
        raise ValueError("acc shape mismatch")
    for t in (out, acc):
        if t is not None and x.numel() and t.data_ptr() == x.data_ptr():
            raise ValueError("act_conv1d_umma: out/acc must not alias x")
    lib = _lib.load()
    _lib.check(lib.hsv_act_conv1d_umma(_p(x), _p(alpha), _p(beta), float(scale), _p(w_packed), _p(bias), _p(residual),
                                       _p(out), _p(acc), acc_mode, B, cin, cout, L, k, d, _stream()),
               "hsv_act_conv1d_umma")
    return out


FUSED_CIN = (16, 32, 64)   # channel counts the activation-producing conv variant takes (single operand chunk)


def pack_convT_weight(w: torch.Tensor, u: int, n_tile: int) -> torch.Tensor:
    """w: folded ConvTranspose1d weight [Cin, Cout, k] -> packed fp16 phase/tap stream."""
    _req(w, "w", ndim=3)
    cin, cout, k = w.shape
    out = torch.empty(cout * cin * k, dtype=torch.float16, device=w.device)
    lib = _lib.load()
    _lib.check(lib.hsv_pack_convT_weight(_p(w), _p(out), cin, cout, k, u, n_tile, _stream()), "hsv_pack_convT_weight")
    _static_data_barrier("pack_convT_weight")
    return out


def conv_transpose1d_umma(a_blk: torch.Tensor, w_packed: torch.Tensor, bias: Optional[torch.Tensor], Lin: int,
                          cin: int, cout: int, k: int, u: int, n_tile: int, add: Optional[torch.Tensor] = None):
    """tcgen05 ConvTranspose1d (polyphase).  Returns fp32 [B, Cout, u*Lin]."""
    _req(a_blk, "a_blk16", torch.float16, 4); _req(w_packed, "w_packed", torch.float16)
    B = a_blk.shape[0]
    if tuple(a_blk.shape) != blk16_shape(B, cin, Lin):
        raise ValueError(f"a_blk16 shape {tuple(a_blk.shape)} does not match Cin={cin}, L={Lin}")
    if w_packed.numel() < cout * cin * k:
        raise ValueError("w_packed size mismatch")
    out = torch.empty(B, cout, u * Lin, dtype=torch.float32, device=a_blk.device)
    if bias is not None:
        _req(bias, "bias")
    if add is not None:
        _req(add, "add", ndim=3)
        if add.shape != out.shape:
            raise ValueError("add shape mismatch")
    lib = _lib.load()
    _lib.check(lib.hsv_conv_transpose1d_umma(_p(a_blk), _p(w_packed), _p(bias), _p(add), _p(out), B, cin, cout, Lin,
                                             k, u, n_tile, _stream()), "hsv_conv_transpose1d_umma")
    return out


def conv1d_direct(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], d: int = 1, pad: int = 0,
                  flags: int = 0, out: Optional[torch.Tensor] = None, valid_len: Optional[torch.Tensor] = None):
    """fp32 Conv1d on CUDA cores.  ``valid_len`` (int32 [B], conv_post shapes only: Cout <= 4, k = 7, pad = 3): item b
    reads x[..., :valid_len[b]] only and its output past that is 0."""
    _req(x, "x", ndim=3); _req(w, "w", ndim=3)
    if bias is not None:
        _req(bias, "bias")
    B, cin, Lin = x.shape
    cout, cin_w, k = w.shape
    if cin_w != cin:
        raise ValueError(f"weight Cin {cin_w} != input Cin {cin}")
    Lout = Lin + 2 * pad - d * (k - 1)
    if out is None:
        if flags & CONV_ADD_OUT:
            raise ValueError("CONV_ADD_OUT needs an out tensor")
        out = torch.empty(B, cout, Lout, dtype=torch.float32, device=x.device)
    else:
        _req(out, "out", ndim=3)
        if tuple(out.shape) != (B, cout, Lout):
            raise ValueError("out shape mismatch")
    _req_len(valid_len, B, x.device)
    lib = _lib.load()
    if valid_len is not None:
        _lib.check(lib.hsv_conv1d_direct_ragged(_p(x), _p(w), _p(bias), _p(valid_len), _p(out), B, cin, cout, Lin, Lout,
                                                k, d, pad, flags, _stream()), "hsv_conv1d_direct_ragged")
    else:
        _lib.check(lib.hsv_conv1d_direct(_p(x), _p(w), _p(bias), _p(out), B, cin, cout, Lin, Lout, k, d, pad, flags,
                                         _stream()), "hsv_conv1d_direct")
    return out


def conv_transpose1d(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], u: int,
                     add: Optional[torch.Tensor] = None):
    _req(x, "x", ndim=3); _req(w, "w", ndim=3)
    B, cin, Lin = x.shape
    cin_w, cout, k = w.shape
    if cin_w != cin:
        raise ValueError(f"weight Cin {cin_w} != input Cin {cin}")
    out = torch.empty(B, cout, u * Lin, dtype=torch.float32, device=x.device)
    if add is not None:
        _req(add, "add", ndim=3)
        if add.shape != out.shape:
            raise ValueError("add shape mismatch")
    if bias is not None:
        _req(bias, "bias")
    lib = _lib.load()
    _lib.check(lib.hsv_conv_transpose1d_direct(_p(x), _p(w), _p(bias), _p(add), _p(out), B, cin, cout, Lin, k, u,
                                               _stream()), "hsv_conv_transpose1d_direct")
    return out


def sr_pre_interp(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], Lout: int,
                  valid_len: Optional[Tuple[torch.Tensor, torch.Tensor]] = None):
    """SpeechSR conv_pre + linear interpolation to Lout.  ``valid_len`` = (len_in, len_out), int32 [B] each: item b is
    interpolated from len_in[b] to len_out[b] samples as if run alone; its output past len_out[b] is 0."""
    _req(x, "x", ndim=3); _req(w, "w", ndim=3)
    B, one, Lin = x.shape
    C = w.shape[0]
    if one != 1 or tuple(w.shape[1:]) != (1, 7):
        raise ValueError("sr_pre_interp expects x [B,1,L] and w [C,1,7]")
    out = torch.empty(B, C, Lout, dtype=torch.float32, device=x.device)
    lib = _lib.load()
    if valid_len is not None:
        vin, vout = valid_len
        _req_len(vin, B, x.device, "valid_len[0]"); _req_len(vout, B, x.device, "valid_len[1]")
        _lib.check(lib.hsv_sr_pre_interp_ragged(_p(x), _p(w), _p(bias), _p(vin), _p(vout), _p(out), B, C, Lin, Lout,
                                                _stream()), "hsv_sr_pre_interp_ragged")
    else:
        _lib.check(lib.hsv_sr_pre_interp(_p(x), _p(w), _p(bias), _p(out), B, C, Lin, Lout, _stream()),
                   "hsv_sr_pre_interp")
    return out


SR_RATIOS = {3: (3, 1), 1.5: (3, 2)}   # SpeechSR scale -> (up, down)


def _req_ratio(ratio):
    if tuple(ratio) not in SR_RATIOS.values():
        raise ValueError(f"ratio must be one of {sorted(SR_RATIOS.values())} (up, down), got {ratio}")
    return tuple(ratio)


def sr_pre_interp_stream(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], Lout: int,
                         valid_len: Tuple[torch.Tensor, torch.Tensor], origin: torch.Tensor, ratio):
    """``sr_pre_interp`` of streaming windows: item b is the window x[b, 0, :valid_len[0][b]] of a stream, at the stream's
    input / output sample origin[b, 0] / origin[b, 1] (int64 [B, 3]; origin[b, 2] = the stream's total length on its last
    window, else -1).  ``ratio`` = (up, down) = (3, 1) or (3, 2).  Outputs are those of the whole stream at the same
    global indices wherever every conv_pre tap lies inside the window (include/hsv.h)."""
    _req(x, "x", ndim=3); _req(w, "w", ndim=3)
    if bias is not None:
        _req(bias, "bias")
    B, one, Lin = x.shape
    C = w.shape[0]
    if one != 1 or tuple(w.shape[1:]) != (1, 7):
        raise ValueError("sr_pre_interp_stream expects x [B,1,L] and w [C,1,7]")
    up, down = _req_ratio(ratio)
    vin, vout = valid_len
    _req_len(vin, B, x.device, "valid_len[0]"); _req_len(vout, B, x.device, "valid_len[1]")
    _req(origin, "origin", torch.int64, 2)
    if tuple(origin.shape) != (B, 3) or origin.device != x.device:
        raise ValueError(f"origin must be int64 [{B}, 3] on {x.device}, got {tuple(origin.shape)} on {origin.device}")
    out = torch.empty(B, C, Lout, dtype=torch.float32, device=x.device)
    lib = _lib.load()
    _lib.check(lib.hsv_sr_pre_interp_stream(_p(x), _p(w), _p(bias), _p(vin), _p(vout), _p(origin), _p(out), B, C, Lin,
                                            Lout, up, down, _stream()), "hsv_sr_pre_interp_stream")
    return out


def sr_stream_window(x_new: torch.Tensor, n_new: torch.Tensor, start: torch.Tensor, end: torch.Tensor,
                     hist: torch.Tensor, state: torch.Tensor, ratio, lookahead: int):
    """One step's windows of S SpeechSR streams (include/hsv.h, ``hsv_sr_stream_window``).  Returns (win [S, H + N],
    valid_len_in [S], valid_len_out [S], origin [S, 3], plan [S, 6]); ``hist`` / ``state`` are only read."""
    _req(x_new, "x_new", ndim=2)
    S, N = x_new.shape
    for t, name in ((n_new, "n_new"), (start, "start"), (end, "end")):
        _req_len(t, S, x_new.device, name)
    _req(hist, "hist", ndim=2); _req(state, "state", torch.int64, 2)
    H = hist.shape[1]
    if hist.shape[0] != S or tuple(state.shape) != (S, 3):
        raise ValueError(f"hist must be [{S}, H] and state [{S}, 3], got {tuple(hist.shape)} and {tuple(state.shape)}")
    if hist.device != x_new.device or state.device != x_new.device:
        raise ValueError("hist and state must be on the device of x_new")
    up, down = _req_ratio(ratio)
    dev = x_new.device
    win = torch.empty(S, H + N, dtype=torch.float32, device=dev)
    vin = torch.empty(S, dtype=torch.int32, device=dev)
    vout = torch.empty(S, dtype=torch.int32, device=dev)
    origin = torch.empty(S, 3, dtype=torch.int64, device=dev)
    plan = torch.empty(S, 6, dtype=torch.int64, device=dev)
    lib = _lib.load()
    _lib.check(lib.hsv_sr_stream_window(_p(x_new), _p(n_new), _p(start), _p(end), _p(hist), _p(state), _p(win), _p(vin),
                                        _p(vout), _p(origin), _p(plan), S, N, H, up, down, int(lookahead), _stream()),
               "hsv_sr_stream_window")
    return win, vin, vout, origin, plan


def sr_stream_emit(y: torch.Tensor, win: torch.Tensor, origin: torch.Tensor, plan: torch.Tensor, hist: torch.Tensor,
                   state: torch.Tensor, cap: int):
    """Copy each stream's newly final outputs of ``y`` [S, Lout] into out [S, cap], and advance ``hist`` / ``state`` in
    place (include/hsv.h, ``hsv_sr_stream_emit``).  Returns (out, n_out int32 [S])."""
    _req(y, "y", ndim=2); _req(win, "win", ndim=2); _req(origin, "origin", torch.int64, 2)
    _req(plan, "plan", torch.int64, 2); _req(hist, "hist", ndim=2); _req(state, "state", torch.int64, 2)
    S, Lout = y.shape
    H, W = hist.shape[1], win.shape[1]
    for t in (win, origin, plan, hist, state):
        if t.shape[0] != S or t.device != y.device:
            raise ValueError(f"every stream tensor must have {S} rows on {y.device}")
    dev = y.device
    out = torch.empty(S, cap, dtype=torch.float32, device=dev)
    n_out = torch.empty(S, dtype=torch.int32, device=dev)
    lib = _lib.load()
    _lib.check(lib.hsv_sr_stream_emit(_p(y), _p(win), _p(origin), _p(plan), _p(hist), _p(state), _p(out), _p(n_out), S,
                                      H, W, Lout, int(cap), _stream()), "hsv_sr_stream_emit")
    return out, n_out


def interp_linear_table(Lin: int, Lout: int, device):
    i0 = torch.empty(Lout, dtype=torch.int32, device=device)
    i1 = torch.empty(Lout, dtype=torch.int32, device=device)
    lam = torch.empty(Lout, dtype=torch.float32, device=device)
    if not i0.is_cuda:
        raise RuntimeError("interp_linear_table: CUDA device required")
    lib = _lib.load()
    _lib.check(lib.hsv_interp_linear_table(Lin, Lout, _p(i0), _p(i1), _p(lam), _stream()), "hsv_interp_linear_table")
    return i0, i1, lam


def nearest_gather(x: torch.Tensor, Lout: int):
    _req(x, "x", ndim=3)
    B, C, Lin = x.shape
    out = torch.empty(B, C, Lout, dtype=torch.float32, device=x.device)
    lib = _lib.load()
    _lib.check(lib.hsv_nearest_gather(_p(x), _p(out), B * C, Lin, Lout, _stream()), "hsv_nearest_gather")
    return out


def add3_bcast(a: torch.Tensor, b: Optional[torch.Tensor], bc: Optional[torch.Tensor], out: Optional[torch.Tensor] = None):
    """out = a + b + bc (bc is [B,C,1], broadcast along L)."""
    _req(a, "a", ndim=3)
    B, C, L = a.shape
    if b is not None:
        _req(b, "b", ndim=3)
        if b.shape != a.shape:
            raise ValueError("b shape mismatch")
    if bc is not None:
        _req(bc, "bc")
        if bc.numel() != B * C:
            raise ValueError("bc must be [B,C,1]")
    if out is None:
        out = torch.empty_like(a)
    lib = _lib.load()
    _lib.check(lib.hsv_add3_bcast(_p(a), _p(b), _p(bc), _p(out), B * C, L, _stream()), "hsv_add3_bcast")
    return out


def peak_norm_pcm16(x: torch.Tensor, s1: float = 32767.0, s2: float = 0.999, per_row: bool = False):
    """int16 PCM of ``x / max|x| * s1 * s2`` (fp32, reference operation order, truncation like numpy's astype).

    x: fp32 [..., L]; leading dims are rows.  ``per_row=False`` uses one peak for the whole tensor
    (inference_plm.py:183-188 / inference_speechsr.py:39-41), ``True`` one per row.  An all-zero row (or tensor, for
    the global peak) has peak 0: 0 / 0 is NaN, and the device's float-to-int conversion makes it 0, so its PCM is all
    zeros (numpy's NaN -> int16 cast is platform-defined).  Returns (pcm int16, peaks fp32)."""
    _req(x, "x")
    if x.dim() < 1:
        raise ValueError("x must have at least one dim")
    L = x.shape[-1]
    rows = x.numel() // L if L else 0
    out = torch.empty(x.shape, dtype=torch.int16, device=x.device)
    peaks = torch.zeros(max(rows, 1), dtype=torch.float32, device=x.device)
    lib = _lib.load()
    _lib.check(lib.hsv_peak_norm_pcm16(_p(x), _p(out), _p(peaks), rows, L, float(s1), float(s2), int(per_row), _stream()),
               "hsv_peak_norm_pcm16")
    return out, (peaks if per_row else peaks[:1])


def peak_norm_pcm16_rows(x: torch.Tensor, s2: torch.Tensor, s1: float = 32767.0):
    """``peak_norm_pcm16(per_row=True)`` with one ``s2`` per row: row b equals ``peak_norm_pcm16(x[b], s1, s2[b])``.
    s2: fp32 CUDA [rows].  Returns (pcm int16, peaks fp32 [rows])."""
    _req(x, "x"); _req(s2, "s2", ndim=1)
    if x.dim() < 1:
        raise ValueError("x must have at least one dim")
    L = x.shape[-1]
    rows = x.numel() // L if L else 0
    if s2.numel() != rows or s2.device != x.device:
        raise ValueError(f"s2: expected {rows} values on {x.device}, got {s2.numel()} on {s2.device}")
    out = torch.empty(x.shape, dtype=torch.int16, device=x.device)
    peaks = torch.zeros(max(rows, 1), dtype=torch.float32, device=x.device)
    _lib.check(_lib.load().hsv_peak_norm_pcm16_rows(_p(x), _p(out), _p(peaks), rows, L, float(s1), _p(s2), _stream()),
               "hsv_peak_norm_pcm16_rows")
    return out, peaks


def resample(x: torch.Tensor, rate: torch.Tensor, valid_len: torch.Tensor, table: torch.Tensor, desc, new_freq: int,
             out_len: int):
    """Kaiser-windowed sinc resampling of a ragged batch to ``new_freq`` (include/hsv.h, ``hsv_resample_ragged``).
    x: fp32 or int16 [B, T]; rate / valid_len: int32 [B] on x's device; table: fp32 [n] (the filters, [K][n] each);
    desc: host rows (rate, o, n, width, K, offset).  Returns (y fp32 [B, out_len], n_out int32 [B])."""
    if not isinstance(x, torch.Tensor) or x.dtype not in (torch.float32, torch.int16):
        raise ValueError("x: expected a float32 or int16 tensor")
    _req(x, "x", x.dtype, 2)
    B, T = x.shape
    _req_len(rate, B, x.device, "rate"); _req_len(valid_len, B, x.device, "valid_len")
    _req(table, "table", ndim=1)
    if table.device != x.device:
        raise ValueError(f"table is on {table.device}, x on {x.device}")
    flat = [int(v) for row in desc for v in row]
    host_desc = (ctypes.c_int32 * len(flat))(*flat)
    y = torch.empty(B, out_len, dtype=torch.float32, device=x.device)
    n_out = torch.empty(B, dtype=torch.int32, device=x.device)
    _lib.check(_lib.load().hsv_resample_ragged(_p(x), int(x.dtype == torch.int16), _p(rate), _p(valid_len), _p(table),
                                               table.numel(), host_desc, len(desc), int(new_freq), _p(y), _p(n_out), B,
                                               T, int(out_len), _stream()), "hsv_resample_ragged")
    return y, n_out


# ----------------------------------------------------------------------------------------------
# frame-rate operators of the step before the vocoder (csrc/frame_ops.cu)
# ----------------------------------------------------------------------------------------------
CONV_SILU_IN = 8
CONV_LRELU001_IN = 16
PACK_MASK, PACK_GATE, PACK_GELU, PACK_MISH = 0, 1, 2, 3
(OP_WN_RES, OP_WN_LAST, OP_GATE_ADD, OP_COUPLE, OP_SAMPLE, OP_MASK, OP_ADD, OP_GLU_RES, OP_MISH, OP_FLIP,
 OP_ADD_BCAST) = range(1, 12)


def _req_vec(t: torch.Tensor, name: str):
    """Per-(batch, channel) vectors may be strided views (e.g. a chunk of the adaLN output): pointer + batch stride."""
    if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype != torch.float32:
        raise RuntimeError(f"{name}: expected a CUDA float32 tensor (no CPU fallback)")
    if t.stride(-1) != 1 and t.shape[-1] != 1:
        raise ValueError(f"{name}: innermost dimension must be dense")


def pack_blk16_act(x: torch.Tensor, buf: torch.Tensor, C: int, mode: int = PACK_MASK, bcast: Optional[torch.Tensor] = None,
                   mask: Optional[torch.Tensor] = None, c_off: int = 0):
    """fp32 [B, >=c_off+C (>=2C for the gate), T] -> fp16 blk16 [C] with a fused activation (hsv_pack_blk16_act);
    channels [c_off, c_off+C) of x are used (the gate: [0, 2C))."""
    _req(x, "x", ndim=3); _req(buf, "buf", torch.float16, 4)
    B, cin, L = x.shape
    if cin < c_off + (2 * C if mode == PACK_GATE else C) or (c_off and mode == PACK_GATE):
        raise ValueError(f"pack_blk16_act: x has {cin} channels, needs {c_off + (2 * C if mode == PACK_GATE else C)}")
    if tuple(buf.shape) != blk16_shape(B, C, L):
        raise ValueError("blk16 buffer shape mismatch")
    if bcast is not None:
        _req(bcast, "bcast")
    if mask is not None:
        _req(mask, "mask")
    lib = _lib.load()
    xp = ctypes.c_void_p(x.data_ptr() + 4 * c_off * L)
    _lib.check(lib.hsv_pack_blk16_act(xp, _p(bcast), _p(mask), _p(buf), B, C, L, mode, cin, _stream()),
               "hsv_pack_blk16_act")
    return buf


def wn_res_pack(x: torch.Tensor, rs: torch.Tensor, mask: Optional[torch.Tensor], output: torch.Tensor, buf: torch.Tensor):
    """WN layer tail fused with the next layer's operand pack: x = (x + rs[:, :C]) * mask (in place), output += rs[:, C:],
    buf = fp16 blk16 operand of the new x."""
    _req(x, "x", ndim=3); _req(rs, "rs", ndim=3); _req(output, "output", ndim=3); _req(buf, "buf", torch.float16, 4)
    B, C, L = x.shape
    if tuple(rs.shape) != (B, 2 * C, L) or tuple(output.shape) != (B, C, L):
        raise ValueError("wn_res_pack: shape mismatch")
    if tuple(buf.shape) != blk16_shape(B, C, L):
        raise ValueError("blk16 buffer shape mismatch")
    if mask is not None:
        _req(mask, "mask")
    _lib.check(_lib.load().hsv_wn_res_pack(_p(x), _p(rs), _p(mask), _p(output), _p(buf), B, C, L, _stream()),
               "hsv_wn_res_pack")
    return buf


LN_ZERO_MASKED = 2


def ln_mod_blk16(x: torch.Tensor, shift: torch.Tensor, scale: torch.Tensor, buf: torch.Tensor, mod_stride: int,
                 mask: Optional[torch.Tensor] = None, eps: float = 1e-6, inmask: bool = False, premask: bool = False,
                 zero_masked: bool = False):
    """LayerNorm over channels (no affine) [* mask] -> x * (1 + scale[b]) + shift[b] -> fp16 blk16.  ``zero_masked``:
    operand rows where mask == 0 are written as zero (rows past an item of a ragged batch)."""
    _req(x, "x", ndim=3); _req_vec(shift, "shift"); _req_vec(scale, "scale"); _req(buf, "buf", torch.float16, 4)
    B, C, L = x.shape
    if tuple(buf.shape) != blk16_shape(B, C, L):
        raise ValueError("blk16 buffer shape mismatch")
    if mask is not None:
        _req(mask, "mask")
    lib = _lib.load()
    if zero_masked and mask is None:
        raise ValueError("ln_mod_blk16: zero_masked needs a mask")
    _lib.check(lib.hsv_ln_mod_blk16(_p(x), _p(shift), _p(scale), _p(mask), _p(buf), B, C, L, float(eps), int(inmask),
                                    int(premask) | (LN_ZERO_MASKED if zero_masked else 0), int(mod_stride), _stream()),
               "hsv_ln_mod_blk16")
    return buf


def gate_ln_mod_blk16(x: torch.Tensor, y: torch.Tensor, gate: torch.Tensor, shift: torch.Tensor, scale: torch.Tensor,
                      buf: torch.Tensor, mod_stride: int, mask: Optional[torch.Tensor] = None, eps: float = 1e-6,
                      premask: bool = False, zero_masked: bool = False):
    """x += gate[b] * y * mask (in place), then ``ln_mod_blk16`` of the new x: one launch.  gate/shift/scale are row views
    of one modulation tensor (batch stride ``mod_stride``); ``zero_masked`` as ``ln_mod_blk16``."""
    _req(x, "x", ndim=3); _req(y, "y", ndim=3); _req_vec(gate, "gate"); _req_vec(shift, "shift"); _req_vec(scale, "scale")
    _req(buf, "buf", torch.float16, 4)
    B, C, L = x.shape
    if tuple(y.shape) != (B, C, L) or tuple(buf.shape) != blk16_shape(B, C, L):
        raise ValueError("gate_ln_mod_blk16: shape mismatch")
    if mask is not None:
        _req(mask, "mask")
    elif zero_masked:
        raise ValueError("gate_ln_mod_blk16: zero_masked needs a mask")
    _lib.check(_lib.load().hsv_gate_ln_mod_blk16(_p(x), _p(y), _p(gate), int(mod_stride), _p(shift), _p(scale), _p(mask),
                                                 _p(buf), B, C, L, float(eps),
                                                 int(premask) | (LN_ZERO_MASKED if zero_masked else 0), int(mod_stride),
                                                 _stream()),
               "hsv_gate_ln_mod_blk16")
    return buf


def frame_op(op: int, a, b=None, c=None, mask=None, out=None, out2=None, B=0, C=0, L=0, s: float = 1.0, cstride: int = 0):
    for t, n in ((a, "a"), (b, "b"), (mask, "mask"), (out, "out"), (out2, "out2")):
        if t is not None:
            _req(t, n)
    if c is not None:
        _req_vec(c, "c")
    lib = _lib.load()
    _lib.check(lib.hsv_frame_op(int(op), _p(a), _p(b), _p(c), _p(mask), _p(out), _p(out2), B, C, L, float(s), int(cstride),
                                _stream()), "hsv_frame_op")


def mha(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, B: int, heads: int, D: int, Tq: int, Tk: int, q_bs: int,
        k_bs: int, v_bs: int, scale: float, prescale_q: bool, lens: Optional[torch.Tensor] = None,
        out_blk: Optional[torch.Tensor] = None, valid_len: Optional[torch.Tensor] = None) -> torch.Tensor:
    """softmax(q k^T * scale) v; q/k/v may be views into one fused [B, 3*heads*D, T] tensor (pass batch strides).
    ``out_blk``: write the result as the fp16 blk16 operand of the conv that follows (tensor-core kernel only) and
    return that buffer instead of a fp32 tensor.  ``valid_len`` (int32 [B], self-attention, not with ``lens``): item b
    is its first valid_len[b] frames as if run alone with Tq = Tk = valid_len[b]; its rows past that are 0."""
    for t, n in ((q, "q"), (k, "k"), (v, "v")):
        if not t.is_cuda or t.dtype != torch.float32:
            raise RuntimeError(f"mha: {n} must be a CUDA float32 tensor")
    if lens is not None:
        _req(lens, "lens", torch.int32)
    lib = _lib.load()
    if valid_len is not None:
        _req_len(valid_len, B, q.device)
        if lens is not None or Tq != Tk:
            raise ValueError("mha: valid_len is per-item self-attention (Tq == Tk, no lens)")
        if out_blk is not None:
            _req(out_blk, "out_blk", torch.float16, 4)
            if tuple(out_blk.shape) != blk16_shape(B, heads * D, Tq):
                raise ValueError("mha: blk16 buffer shape mismatch")
            out = out_blk
        else:
            out = torch.empty(B, heads * D, Tq, dtype=torch.float32, device=q.device)
        _lib.check(lib.hsv_mha_ragged(_p(q), _p(k), _p(v), _p(out), int(out_blk is not None), None, _p(valid_len), B, heads,
                                      D, Tq, Tk, int(q_bs), int(k_bs), int(v_bs), float(scale), int(prescale_q), _stream()),
                   "hsv_mha_ragged")
        return out
    if out_blk is not None:
        _req(out_blk, "out_blk", torch.float16, 4)
        if tuple(out_blk.shape) != blk16_shape(B, heads * D, Tq):
            raise ValueError("mha: blk16 buffer shape mismatch")
        _lib.check(lib.hsv_mha_blk16(_p(q), _p(k), _p(v), _p(out_blk), _p(lens), B, heads, D, Tq, Tk, int(q_bs), int(k_bs),
                                     int(v_bs), float(scale), int(prescale_q), _stream()), "hsv_mha_blk16")
        return out_blk
    out = torch.empty(B, heads * D, Tq, dtype=torch.float32, device=q.device)
    _lib.check(lib.hsv_mha(_p(q), _p(k), _p(v), _p(out), _p(lens), B, heads, D, Tq, Tk, int(q_bs), int(k_bs), int(v_bs),
                           float(scale), int(prescale_q), _stream()), "hsv_mha")
    return out


def conv1d_c1_strided(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], stride: int, pad: int,
                      mask: Optional[torch.Tensor] = None, valid_len: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Conv1d(1, Cout, k, stride, pad) * mask.  ``valid_len`` (int32 [B], output frames): item b reads
    x[b, 0, :stride * valid_len[b]] only, as its own run with that many samples, and its output past valid_len[b] is 0."""
    _req(x, "x", ndim=3); _req(w, "w", ndim=3)
    B, one, Lin = x.shape
    cout, one_w, k = w.shape
    if one != 1 or one_w != 1:
        raise ValueError("conv1d_c1_strided: single input channel only")
    Lout = (Lin + 2 * pad - k) // stride + 1
    out = torch.empty(B, cout, Lout, dtype=torch.float32, device=x.device)
    lib = _lib.load()
    if valid_len is not None:
        _req_len(valid_len, B, x.device)
        _lib.check(lib.hsv_conv1d_c1_strided_ragged(_p(x), _p(w), _p(bias), _p(mask), _p(valid_len), _p(out), B, cout, Lin,
                                                    Lout, k, stride, pad, _stream()), "hsv_conv1d_c1_strided_ragged")
    else:
        _lib.check(lib.hsv_conv1d_c1_strided(_p(x), _p(w), _p(bias), _p(mask), _p(out), B, cout, Lin, Lout, k, stride, pad,
                                             _stream()), "hsv_conv1d_c1_strided")
    return out


def masked_mean(x: torch.Tensor, mask: Optional[torch.Tensor], valid_len: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x.sum(2) / mask.sum(2) over all L frames; ``valid_len`` (int32 [B]): item b's mean over its first valid_len[b]
    frames, summed in the order of its own run (the mask is then not read).

    Empty items are not rejected: an item with valid_len 0 gives NaN (0 / 0, the mean of its own, empty run, as
    ``torch.mean`` of an empty tensor); without ``valid_len`` an all-zero mask row gives x.sum(2) / 0 as the reference
    does (+-inf, or NaN where the sum is 0)."""
    _req(x, "x", ndim=3)
    B, C, L = x.shape
    out = torch.empty(B, C, dtype=torch.float32, device=x.device)
    lib = _lib.load()
    if valid_len is not None:
        _req_len(valid_len, B, x.device)
        _lib.check(lib.hsv_masked_mean_ragged(_p(x), _p(mask), _p(valid_len), _p(out), B, C, L, _stream()),
                   "hsv_masked_mean_ragged")
    else:
        _lib.check(lib.hsv_masked_mean(_p(x), _p(mask), _p(out), B, C, L, _stream()), "hsv_masked_mean")
    return out


def _req_seeds(seeds: torch.Tensor, B: Optional[int] = None):
    _req(seeds, "seeds", torch.int64, 1)
    if B is not None and seeds.numel() != B:
        raise ValueError(f"seeds: expected {B} elements, got {seeds.numel()}")


def seeded_normal(seeds: torch.Tensor, C: int, T: int, valid_len: Optional[torch.Tensor] = None) -> torch.Tensor:
    """fp32 [B, C, T] standard normals; the value at (b, c, t) depends on (seeds[b], c, t) only (csrc/noise.cu: Philox4x32-10
    + Box-Muller, the project's own stream, not torch's ``randn``).  seeds: int64 CUDA [B].  ``valid_len`` (int32 [B]):
    0 at t >= valid_len[b]."""
    _req_seeds(seeds)
    B = seeds.numel()
    _req_len(valid_len, B, seeds.device)
    out = torch.empty(B, C, T, dtype=torch.float32, device=seeds.device)
    _lib.check(_lib.load().hsv_seeded_normal(_p(seeds), _p(out), B, int(C), int(T), _p(valid_len), _stream()),
               "hsv_seeded_normal")
    return out


def sample_ragged(stats: torch.Tensor, s, valid_len: Optional[torch.Tensor] = None, eps: Optional[torch.Tensor] = None,
                  seeds: Optional[torch.Tensor] = None) -> torch.Tensor:
    """z = (m + n * exp(logs) * s[b]) for stats = [B, 2C, T] (m | logs), the same bits as ``frame_op(OP_SAMPLE)`` fed with
    the same noise n; 0 at t >= valid_len[b] (int32 [B]), where nothing is read.  n: ``eps`` [B, C, T] or, from
    ``seeds`` (int64 [B]), ``seeded_normal(seeds, C, T)`` generated in registers (no noise tensor).  ``s``: a float or a
    fp32 CUDA tensor [B]."""
    _req(stats, "stats", ndim=3)
    B, C2, T = stats.shape
    C = C2 // 2
    if C2 % 2:
        raise ValueError(f"stats must have 2C channels, got {C2}")
    if (eps is None) == (seeds is None):
        raise ValueError("sample_ragged: pass exactly one of eps and seeds")
    if eps is not None:
        _req(eps, "eps", ndim=3)
        if tuple(eps.shape) != (B, C, T):
            raise ValueError(f"eps must have shape {(B, C, T)}, got {tuple(eps.shape)}")
    else:
        _req_seeds(seeds, B)
    _req_len(valid_len, B, stats.device)
    svec = None
    if isinstance(s, torch.Tensor):
        _req(s, "s", ndim=1)
        if s.numel() != B:
            raise ValueError(f"s: expected {B} elements, got {s.numel()}")
        svec, s = s, 0.0
    for t, n in ((eps, "eps"), (seeds, "seeds"), (svec, "s")):
        if t is not None and t.device != stats.device:
            raise ValueError(f"{n}: on {t.device}, stats is on {stats.device}")
    out = torch.empty(B, C, T, dtype=torch.float32, device=stats.device)
    _lib.check(_lib.load().hsv_sample_ragged(_p(stats), _p(eps), _p(seeds), _p(svec), float(s), _p(valid_len), _p(out), B,
                                             C, T, _stream()), "hsv_sample_ragged")
    return out


def sinegen(f0: torch.Tensor, hop: int, sample_rate: float, harmonics: int = 8, amp: float = 0.1):
    """Harmonic sine source from a frame-rate f0 track (Hz, <= 0 = unvoiced): returns (sines [B, harmonics, T*hop],
    voiced mask [B, 1, T*hop]).  64-bit fixed-point phase accumulation: no drift over long utterances."""
    _req(f0, "f0", ndim=2)
    B, T = f0.shape
    L = T * hop
    out = torch.empty(B, harmonics, L, dtype=torch.float32, device=f0.device)
    uv = torch.empty(B, 1, L, dtype=torch.float32, device=f0.device)
    lib = _lib.load()
    ws = torch.empty(max(1, int(lib.hsv_sinegen_workspace(B, T, hop)) // 8), dtype=torch.int64, device=f0.device)
    _lib.check(lib.hsv_sinegen(_p(f0), _p(out), _p(uv), _p(ws), B, T, hop, float(sample_rate), harmonics, float(amp),
                               _stream()), "hsv_sinegen")
    return out, uv


MHA_VARIANT = [0]


def set_mha_variant(v: int):
    """Test hook: 0 = tensor-core attention (default), 1 = the fp32 CUDA-core kernel."""
    _lib.check(_lib.load().hsv_set_mha_variant(int(v)), "hsv_set_mha_variant")
    MHA_VARIANT[0] = int(v)


def set_act_variant(v: int):
    """Bring-up / test aid: bits 0..1 = tensor-core activation policy (0 auto, 1 off, 2 forced), bits 8.. = forced run
    length of the CUDA-core kernel."""
    _lib.load().hsv_set_act_variant(int(v))


def set_umma_debug(flags: int):
    _lib.load().hsv_set_umma_debug(int(flags))


LAUNCH_CONV, LAUNCH_ACT, LAUNCH_MHA, LAUNCH_DIRECT = 0, 1, 2, 3
_LAUNCH_FIELDS = {
    LAUNCH_CONV: ("kind", "msub", "warps", "vec_epi", "nphase", "n_tile", "stages", "G", "resident", "nabuf",
                  "grid_x", "grid_y", "grid_z", "blk_mode", "launches"),
    LAUNCH_ACT: ("R", "mma", "out_mode", "has_valid_len", "launches"),
    LAUNCH_MHA: ("kernel", "D", "out_mode", "has_lens", "has_valid_len", "prescale", "kv16", "q16", "key_tiles",
                 "grid_x", "grid_y", "grid_z", "launches"),
    LAUNCH_DIRECT: ("kernel", "flags", "has_valid_len", "grid_x", "grid_y", "grid_z", "launches"),
}
CONV_ONE_TILE, CONV_PERSISTENT, CONV_FUSED_ACT, CONV_OPERAND_OUT = range(4)
# LAUNCH_DIRECT kernels (csrc/conv_direct.cu)
DIRECT_VECDOT, DIRECT_ROWDOT, DIRECT_THIN_VEC, DIRECT_THIN_SMEM, DIRECT_THIN, DIRECT_TILED, DIRECT_CONVT = range(7)


def last_launch_config(family: int) -> Dict[str, int]:
    """Test hook: the variant the most recent host-side launch decision of a kernel family chose (``LAUNCH_CONV``: the
    tcgen05 conv, ``LAUNCH_ACT``: the fused activation, ``LAUNCH_MHA``: attention, ``LAUNCH_DIRECT``: the CUDA-core
    conv / ConvTranspose of conv_direct.cu), as a dict of the fields
    ``hsv_last_launch_config`` fills.
    Read-only; needs no GPU."""
    names = _LAUNCH_FIELDS[family]
    buf = (ctypes.c_int * len(names))()
    n = _lib.load().hsv_last_launch_config(int(family), ctypes.cast(buf, ctypes.c_void_p), len(names))
    if n != len(names):
        raise _lib.HsvError(f"hsv_last_launch_config({family}) returned {n}, expected {len(names)}")
    return dict(zip(names, buf))
