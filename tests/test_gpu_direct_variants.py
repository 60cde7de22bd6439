"""The fp32 CUDA-core convolutions against a float64 reference at every kernel their dispatch selects.

``hsv_conv1d_direct[_ragged]`` (csrc/conv_direct.cu) picks one of six kernels from the shape, the flags and the 16-byte
alignment of x, w and out; ``hsv_conv_transpose1d_direct`` has one.  They compute the last op of every waveform
(conv_post + tanh), the PitchPredictor's conv_post (leaky_relu(0.01) input), every cond / adaLN vector (1x1 conv,
SiLU input) and the fallbacks of ``modules._dense_conv`` / ``_dense_convT`` for channel counts that are not multiples
of 16.  Every case reads back, through ``ops.last_launch_config(ops.LAUNCH_DIRECT)``, the kernel it ran and asserts it
is the one it meant to run; its key ``direct:{kernel}:{flags}:{full|ragged}`` goes into ``VERIFIED``.

Reference: float64 on the device from the kernel's fp32 inputs and weights, in the kernels' order of operations: the
input flag, the conv, the bias, tanh, then ``+ out_prev`` (ADD_OUT adds after tanh).  Bound per output: see
``_bound``.  A CPU test shows that the bound accepts fp32 emulations of the kernels' two summation orders and rejects a
shifted tap, the wrong leaky_relu slope, tanh after the add, and fp16 inputs or weights.

(a) the six conv kernels x every input flag x TANH x ADD_OUT, each kernel forced through the dispatch rule (alignment
    by a view one float into a larger buffer).
(b) shape edges per kernel: CTA tiles, staging chunks, the Lout <= 8 switch, the vecdot lane stride, KMAX / HALO_MAX.
(c) the ragged thin kernels (thin_vec, thin_smem) against fp64: the <= 8-step short items, the float4 straddling
    valid_len at both window edges, clamping; inputs past valid_len are NaN, outputs there must be exactly 0.
(d) the direct ConvTranspose at every (k, u) the C-ABI accepts with u <= 8, at the channel counts it exists for.
(e) sr_pre_interp, conv1d_c1_strided and weight_norm_fold, full and ragged.
(f) production conv_post shapes, spot-checked on windows at both ends and across 512-step tile edges.
(g) census: every CUDA-core conv launch of the benchmark workloads and of ragged / per-item batches is in VERIFIED.
"""
import argparse
import math
import os
import sys
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

DEV = "cuda:0"
U32 = 2.0 ** -24            # unit roundoff of fp32

NONE, LRELU, TANH, ADD, SILU, LRELU001 = 0, 1, 2, 4, 8, 16     # ops.CONV_* (hsv.h HSV_CONV_*)
IN_FLAGS = (NONE, LRELU, LRELU001, SILU)
FLAG_SETS = [f | t | a for f in IN_FLAGS for t in (0, TANH) for a in (0, ADD)]
KERNELS = ("vecdot", "rowdot", "thin_vec", "thin_smem", "thin", "tiled", "convT")   # record field "kernel" 0..6


def flag_name(flags):
    names = [n for bit, n in ((LRELU, "lrelu"), (LRELU001, "lrelu001"), (SILU, "silu"), (TANH, "tanh"), (ADD, "add"))
             if flags & bit]
    return "+".join(names) or "none"


def direct_key(c):
    """Key of a launch from its ``last_launch_config(LAUNCH_DIRECT)`` record."""
    return f"direct:{KERNELS[c['kernel']]}:{flag_name(c['flags'])}:{'ragged' if c['has_valid_len'] else 'full'}"


def _key(kernel, flags, ragged=False):
    return f"direct:{kernel}:{flag_name(flags)}:{'ragged' if ragged else 'full'}"


# ----------------------------------------------------------------------------------------------
# reference and bound
# ----------------------------------------------------------------------------------------------
LAMBDA = 8.0
# |fp32 flag - fp64 flag| <= FLAG_U[flag] * u * |f(x)|: leaky_relu multiplies by 0.1f / 0.01f (0.25 / 0.375 u away from
# 0.1 / 0.01) and rounds (0.5 u); SiLU v / (1 + expf(-v)): expf within 2 ulp (4 u), the add and the division 0.5 u each
FLAG_U = {NONE: 0.0, LRELU: 1.0, LRELU001: 1.0, SILU: 6.0}


def _flag64(x, flags):
    if flags & LRELU:
        return torch.where(x > 0, x, 0.1 * x)
    if flags & LRELU001:
        return torch.where(x > 0, x, 0.01 * x)
    if flags & SILU:
        return x * torch.sigmoid(x)
    return x


def _bound(S, b_abs, n, flags, y_tanh, y_out):
    """Bound of |fp32 kernel - fp64 reference| per output.

    S = sum_i |w_i f(x_i)| over the n products of the output (taps outside the input count too), b_abs = |bias|.
    - The sum: the kernels add n products and the bias in fp32, as one fmaf chain (ci outer, tap inner) or as lane
      chains plus a shuffle tree.  Each rounding is a relative error <= u of a partial sum; modelled as independent
      zero-mean errors, the total is below LAMBDA sqrt(n) u (S + |b|) with LAMBDA = 8 well past the tail, for both
      orders.  At conv_post's n = 224 that is 120 u S; fp16 inputs or weights err by ~2^-12 |w f(x)| per product.
      test_bound_accepts_fp32_orders_and_rejects_mutants measures both: the fp32 orders stay below 0.1 of the
      bound, fp16 operands exceed it more than 10-fold.
    - The flag's own fp32 error, FLAG_U u |f(x)| per input, adds at most FLAG_U u S.
    - tanh: |tanh'| <= 1 carries the error through; tanhf adds its own 2 ulp <= 4 u |tanh|.
    - ADD_OUT rounds the sum once: u |y|."""
    fu = FLAG_U[flags & (LRELU | LRELU001 | SILU)]
    tol = LAMBDA * math.sqrt(n) * U32 * (S + b_abs) + fu * U32 * S
    if flags & TANH:
        tol = tol + 4 * U32 * y_tanh.abs()
    if flags & ADD:
        tol = tol + U32 * y_out.abs()
    return tol


def conv_ref(x, w, bias, d, pad, flags, prev=None):
    """float64 reference of conv1d_direct and its bound: (ref, tol), [B, Cout, Lout].  Any device; x without NaN."""
    Cin, k = w.shape[1], w.shape[2]
    fx = _flag64(x.double(), flags)
    w64 = w.double()
    y = F.conv1d(fx, w64, None, padding=pad, dilation=d)
    S = F.conv1d(fx.abs(), w64.abs(), None, padding=pad, dilation=d)
    b64 = bias.double()[None, :, None] if bias is not None else torch.zeros_like(y[:1, :, :1])
    y = y + b64
    t = torch.tanh(y) if flags & TANH else y
    out = t + prev.double() if flags & ADD else t
    return out, _bound(S, b64.abs(), Cin * k + 1, flags, t, out)


def _excess(got, ref, tol):
    """max err / tol (0 where both are 0); NaN in ``got`` counts as infinite."""
    err = (got.double() - ref).abs()
    r = torch.where(err == 0, torch.zeros_like(err), err / tol)
    return float(torch.nan_to_num(r, nan=float("inf")).max()) if r.numel() else 0.0


def _check(got, ref, tol, where):
    r = _excess(got, ref, tol)
    assert r <= 1.0, (where, r)
    return r


# ----------------------------------------------------------------------------------------------
# CPU: the bound accepts the kernels' fp32 orders and rejects the mutants
# ----------------------------------------------------------------------------------------------
def _fma(a, b, c):
    """fmaf on the CPU: the fp32 product is exact in float64; one rounding of the sum (a double rounding is rare)."""
    return (a.double() * b.double() + c.double()).float()


def _flag32(x, flags, slope001=0.01):
    if flags & LRELU:
        return torch.where(x > 0, x, torch.tensor(0.1, dtype=torch.float32) * x)
    if flags & LRELU001:
        return torch.where(x > 0, x, torch.tensor(slope001, dtype=torch.float32) * x)
    if flags & SILU:
        return x / (1 + torch.exp(-x))
    return x


def _emulate(x, w, bias, pad, flags, prev, order="chain", shift_tap=None, slope001=0.01, tanh_after_add=False,
             half_x=False, half_w=False):
    """fp32 conv1d_direct (d = 1) on the CPU in a kernel's order: ``chain`` = one fmaf chain per output, ci outer and
    tap inner (thin, thin_smem, thin_vec, tiled); ``warp`` = 32 lane chains over r = ci * k + j, r = lane + 32 m,
    then the xor-shuffle tree (rowdot, short ragged items).  The keyword arguments make the mutants."""
    B, Cin, L = x.shape
    Cout, _, k = w.shape
    Lout = L + 2 * pad - (k - 1)
    if half_x:
        x = x.half().float()
    if half_w:
        w = w.half().float()
    xp = F.pad(_flag32(x, flags, slope001), (pad, pad + 1))

    def term(ci, j):
        s = j + (1 if j == shift_tap else 0)
        return w[:, ci, j][None, :, None], xp[:, ci, None, s:s + Lout]

    if order == "chain":
        acc = torch.zeros(B, Cout, Lout)
        for ci in range(Cin):
            for j in range(k):
                acc = _fma(*term(ci, j), acc)
    else:
        lanes = []
        for lane in range(32):
            a = torch.zeros(B, Cout, Lout)
            for r in range(lane, Cin * k, 32):
                a = _fma(*term(r // k, r % k), a)
            lanes.append(a)
        o = 16
        while o:
            lanes = [lanes[i] + lanes[i ^ o] for i in range(32)]
            o >>= 1
        acc = lanes[0]
    y = acc + bias[None, :, None] if bias is not None else acc
    if tanh_after_add:
        if flags & ADD:
            y = y + prev
        return torch.tanh(y) if flags & TANH else y
    if flags & TANH:
        y = torch.tanh(y)
    if flags & ADD:
        y = y + prev
    return y


def _inputs(B, Cin, Cout, L, k, gen, wscale=1.0):
    """x crossing zero with both signs (|x| up to ~40: SiLU saturates, both leaky slopes matter), w of unit gain x
    wscale, bias, out_prev."""
    x = torch.randn(B, Cin, L, generator=gen) * 2.0
    big = torch.rand(B, Cin, L, generator=gen) < 0.05
    x = torch.where(big, x * 15.0, x)
    w = torch.randn(Cout, Cin, k, generator=gen) * (wscale / math.sqrt(Cin * k))
    bias = torch.randn(Cout, generator=gen) * 0.5
    prev = torch.randn(B, Cout, L + 16, generator=gen)      # cut to Lout by the caller
    return x, w, bias, prev


@pytest.mark.parametrize("order,Cin,k,L", [("chain", 32, 7, 700), ("chain", 16, 7, 700), ("warp", 256, 1, 1),
                                           ("warp", 32, 7, 8)])
def test_bound_accepts_fp32_orders_and_rejects_mutants(order, Cin, k, L):
    """At conv_post's n = 32 x 7 = 224 (and the vocoder's 16 x 7, the cond vector's 256 x 1, a short conv_post row):
    the fp32 emulation of the kernel's order is within the bound for every flag set; each mutant is outside it."""
    B, Cout = (2, 2) if L > 8 else (64, 16)
    pad = (k - 1) // 2
    gen = torch.Generator().manual_seed(Cin * k + L)
    x, w, bias, prev = _inputs(B, Cin, Cout, L, k, gen, wscale=2.0)
    Lout = L + 2 * pad - (k - 1)
    prev = prev[:, :, :Lout]
    ratios = {}
    for flags in FLAG_SETS:
        ref, tol = conv_ref(x, w, bias, 1, pad, flags, prev)
        r = _excess(_emulate(x, w, bias, pad, flags, prev, order), ref, tol)
        assert r <= 1.0, (flag_name(flags), r)
        ratios[flag_name(flags)] = r
    mutants = {
        "tap shifted by one": (NONE, dict(shift_tap=k // 2)) if k > 1 else None,
        "lrelu001 slope 0.1": (LRELU001, dict(slope001=0.1)),
        "tanh after add": (TANH | ADD, dict(tanh_after_add=True)),
        "fp16 inputs": (NONE, dict(half_x=True)),
        "fp16 weights": (NONE, dict(half_w=True)),
        "fp16 inputs, silu+tanh": (SILU | TANH, dict(half_x=True)),
    }
    out = {}
    for name, m in mutants.items():
        if m is None:
            continue
        flags, kw = m
        ref, tol = conv_ref(x, w, bias, 1, pad, flags, prev)
        out[name] = _excess(_emulate(x, w, bias, pad, flags, prev, order, **kw), ref, tol)
    print(f"\n[bound] {order} n={Cin * k}: fp32 order worst {max(ratios.values()):.3f}; mutants "
          + ", ".join(f"{n} {r:.1f}" for n, r in out.items()))
    assert all(r > 1.0 for r in out.values()), out


# ----------------------------------------------------------------------------------------------
# GPU helpers
# ----------------------------------------------------------------------------------------------
def _placed(t, off):
    """A contiguous copy of t on the device whose data starts ``off`` floats into a larger buffer (off = 1: not 16-byte
    aligned)."""
    buf = torch.zeros(t.numel() + 8, dtype=t.dtype, device=DEV)
    v = buf[off:off + t.numel()].view(t.shape)
    v.copy_(t)
    return v


def _grid(kernel, B, Cout, Lout):
    if kernel in ("vecdot", "rowdot"):
        return ((B * Cout * (Lout if kernel == "rowdot" else 1) * 32 + 255) // 256, 1, 1)
    if kernel in ("thin_vec", "thin_smem"):
        return (-(-Lout // 512), B, 1)
    if kernel == "thin":
        return (min(max(1, -(-(B * Lout) // 256)), 148 * 32), 1, 1)
    return (-(-Lout // 64), -(-Cout // 32), B)


def _run_direct(ops, x, w, bias, d, pad, flags, prev, xo=0, wo=0, oo=0, valid_len=None):
    """Launch conv1d_direct on x / w / out placed at the given float offsets; returns (out, record)."""
    Lout = prev.shape[-1]
    out = _placed(prev if flags & ADD else torch.full_like(prev, float("nan")), oo)
    before = ops.last_launch_config(ops.LAUNCH_DIRECT)["launches"]
    ops.conv1d_direct(_placed(x, xo), _placed(w, wo), bias, d=d, pad=pad, flags=flags, out=out, valid_len=valid_len)
    rec = ops.last_launch_config(ops.LAUNCH_DIRECT)
    assert rec["launches"] == before + 1, rec
    assert out.shape[-1] == Lout
    return out, rec


def _case(ops, kernel, B, Cin, Cout, L, k, d, pad, flags, seed, xo=0, wo=0, oo=0):
    """One launch against fp64; asserts the kernel, flags and grid it ran.  Returns the key and error / bound."""
    gen = torch.Generator().manual_seed(seed)
    x, w, bias, prev = _inputs(B, Cin, Cout, L, k, gen, wscale=2.0)
    Lout = L + 2 * pad - d * (k - 1)
    x, w, bias, prev = x.to(DEV), w.to(DEV), bias.to(DEV), prev[:, :, :Lout].contiguous().to(DEV)
    got, rec = _run_direct(ops, x, w, bias, d, pad, flags, prev, xo, wo, oo)
    where = (kernel, B, Cin, Cout, L, k, d, pad, flag_name(flags), xo, wo, oo)
    assert (KERNELS[rec["kernel"]], rec["flags"], rec["has_valid_len"]) == (kernel, flags, 0), (where, rec)
    assert (rec["grid_x"], rec["grid_y"], rec["grid_z"]) == _grid(kernel, B, Cout, Lout), (where, rec)
    ref, tol = conv_ref(x, w, bias, d, pad, flags, prev)
    return direct_key(rec), _check(got, ref, tol, where)


# ----------------------------------------------------------------------------------------------
# (a) the six kernels x every flag set
# ----------------------------------------------------------------------------------------------
# kernel: (B, Cin, Cout, L, k, d, pad, x offset, w offset, out offset), forced through the dispatch rule
KERNEL_SHAPES = {
    "vecdot": (3, 64, 40, 1, 1, 1, 0, 0, 0, 0),           # k = 1, Lin = 1, pad 0, Cin % 4 = 0, aligned x and w
    "rowdot": (2, 24, 6, 5, 3, 1, 1, 0, 0, 0),            # Lout = 5 <= 8
    "thin_vec": (2, 20, 3, 1100, 7, 1, 3, 0, 0, 0),       # Cout <= 4, k 7, pad 3, Lin % 4 = 0, aligned x and out
    "thin_smem": (2, 20, 3, 1100, 7, 1, 3, 1, 0, 0),      # the same with x one float off 16-byte alignment
    "thin": (2, 12, 2, 300, 5, 2, 4, 0, 0, 0),            # Cout <= 4, k != 7
    "tiled": (2, 12, 40, 150, 3, 1, 1, 0, 0, 0),          # everything else
}


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", list(KERNEL_SHAPES))
def test_kernel_flags_vs_fp64(hsv, kernel):
    B, Cin, Cout, L, k, d, pad, xo, wo, oo = KERNEL_SHAPES[kernel]
    worst = 0.0
    for i, flags in enumerate(FLAG_SETS):
        key, r = _case(hsv.ops, kernel, B, Cin, Cout, L, k, d, pad, flags, 100 * i + len(kernel), xo, wo, oo)
        assert key == _key(kernel, flags), key
        worst = max(worst, r)
    print(f"\n[parity] direct {kernel}: 16 flag sets, worst error / bound {worst:.3f}")


# ----------------------------------------------------------------------------------------------
# (b) shape edges per kernel: (kernel, B, Cin, Cout, L, k, d, pad, x offset, w offset, out offset)
# ----------------------------------------------------------------------------------------------
EDGE_CASES = []
# thin_vec: Lout = 512 m + r (r = 4, 508), Lin % 4 = 0; Cin across the 16-channel staging chunk; Cout 1-4
for i, (Cin, L) in enumerate(zip((1, 15, 16, 17, 33), (516, 1020, 1532, 2052, 2556))):
    EDGE_CASES.append(("thin_vec", 2, Cin, 1 + i % 4, L, 7, 1, 3, 0, 0, 0))
EDGE_CASES.append(("thin_vec", 1, 33, 4, 1536 + 508, 7, 1, 3, 0, 1, 0))     # a misaligned w does not matter
# thin_smem: Lout = 512 m + r (r = 1, 511, and 4 / 508 misaligned), Lin % 4 = 1, 2, 3; misaligned x or out; pad != 3
for i, (Cin, L, xo, oo) in enumerate(((1, 513, 0, 0), (15, 1535, 0, 0), (16, 1026, 0, 0), (17, 2047, 0, 0),
                                      (33, 1531, 0, 0), (16, 516, 1, 0), (33, 1020, 0, 1), (17, 9, 0, 0))):
    EDGE_CASES.append(("thin_smem", 2, Cin, 1 + i % 4, L, 7, 1, 3, xo, 0, oo))
for pad, L in ((0, 518), (1, 1027), (6, 506), (2, 13)):                        # Lout = L + 2 pad - 6 != Lin
    EDGE_CASES.append(("thin_smem", 2, 17, 2, L, 7, 1, pad, 0, 0, 0))
# rowdot: Lout 1 and 8 (k * Cin below, at and above one warp of products); the vecdot shapes when misaligned or
# Cin % 4 != 0; Lout = 9 on the other side of the switch below
EDGE_CASES += [("rowdot", 3, 5, 7, 1, 3, 1, 1, 0, 0, 0), ("rowdot", 2, 40, 9, 8, 5, 2, 4, 0, 0, 0),
               ("rowdot", 2, 32, 1, 8, 7, 1, 3, 0, 0, 0), ("rowdot", 2, 4, 3, 8, 1, 1, 0, 0, 0, 0),
               ("rowdot", 2, 64, 5, 1, 1, 1, 0, 1, 0, 0), ("rowdot", 2, 64, 5, 1, 1, 1, 0, 0, 1, 0),
               ("rowdot", 2, 62, 5, 1, 1, 1, 0, 0, 0, 0), ("vecdot", 2, 256, 3, 1, 1, 1, 0, 0, 0, 1),
               ("tiled", 2, 40, 9, 9, 5, 2, 4, 0, 0, 0), ("thin", 2, 32, 2, 9, 3, 1, 1, 0, 0, 0),
               ("thin_smem", 2, 32, 1, 9, 7, 1, 3, 0, 0, 0)]
# vecdot (whose out may be misaligned, above): Cin across the 128-float4 stride of the lane loop
EDGE_CASES += [("vecdot", 2, Cin, 1 + Cin % 7, 1, 1, 1, 0, 0, 0, 0) for Cin in (4, 256, 512, 516, 1024, 1028)]
# thin: d > 1, k != 7 (k = 1, 16: KMAX; (k - 1) d = 60 / 64: HALO_MAX)
EDGE_CASES += [("thin", 2, 3, 4, 700, 5, 3, 6, 0, 0, 0), ("thin", 2, 9, 2, 300, 7, 2, 6, 0, 0, 0),
               ("thin", 2, 16, 1, 20, 1, 1, 0, 0, 0, 0), ("thin", 1, 5, 3, 200, 16, 4, 30, 0, 0, 0),
               ("thin", 1, 4, 1, 150, 5, 16, 32, 0, 0, 0)]
# tiled: Cout across the 32-channel tile, Cin across the 8-channel chunk, Lout around the 64-step tile,
# (k - 1) d = 64 (HALO_MAX) and k = 16 (KMAX)
for i, (Cout, Cin, L) in enumerate(((5, 1, 63), (31, 7, 64), (32, 8, 65), (33, 9, 129), (33, 1, 128), (5, 9, 191))):
    EDGE_CASES.append(("tiled", 2, Cin, Cout, L, 3, 1, 1, i % 2, 0, i % 3 == 2))
EDGE_CASES += [("tiled", 2, 9, 33, 130, 5, 16, 32, 0, 0, 0), ("tiled", 2, 7, 31, 100, 16, 1, 7, 0, 0, 0),
               ("tiled", 1, 9, 40, 70, 9, 8, 32, 0, 0, 0), ("tiled", 1, 3, 6, 66, 16, 4, 30, 0, 0, 0)]


def _edge_id(c):
    return f"{c[0]}-B{c[1]}-ci{c[2]}-co{c[3]}-L{c[4]}-k{c[5]}d{c[6]}p{c[7]}-o{c[8]}{c[9]}{int(c[10])}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", EDGE_CASES, ids=[_edge_id(c) for c in EDGE_CASES])
def test_shape_edges_vs_fp64(hsv, case):
    kernel, B, Cin, Cout, L, k, d, pad, xo, wo, oo = case
    seed = zlib.crc32(_edge_id(case).encode())
    for flags in (TANH | ADD, LRELU001, SILU | TANH):
        key, r = _case(hsv.ops, kernel, B, Cin, Cout, L, k, d, pad, flags, seed, xo, wo, int(oo))
        assert key == _key(kernel, flags), key


# ----------------------------------------------------------------------------------------------
# (c) the ragged thin kernels against fp64
# ----------------------------------------------------------------------------------------------
RAGGED_L = 2048


def _ragged_lens(L):
    """0 / 1 / 7 / 8 / 9 (the short-item switch), Lv % 4 = 1, 2, 3 at t0 - 4 and t0 + 4 of the 512-step tiles at
    512 and 1024 (the straddling float4 at each window edge), L - 1, L, a negative and a too-large value."""
    lens = [0, 1, 7, 8, 9]
    for t0 in (512, 1024):
        lens += [t0 - 4 + r for r in (1, 2, 3)] + [t0 + 4 + r for r in (1, 2, 3)]
    return lens + [L - 1, L, -5, L + 100]


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,L,xo", [("thin_vec", RAGGED_L, 0), ("thin_smem", RAGGED_L, 1),
                                         ("thin_smem", RAGGED_L - 3, 0)])
def test_ragged_thin_vs_fp64(hsv, kernel, L, xo):
    ops = hsv.ops
    lens = _ragged_lens(L)
    B, Cin, worst = len(lens), 33, 0.0
    vl = torch.tensor(lens, dtype=torch.int32, device=DEV)
    clamp = [min(max(n, 0), L) for n in lens]
    for i, flags in enumerate(FLAG_SETS):
        Cout = 1 + i % 4
        gen = torch.Generator().manual_seed(L + 17 * i)
        x, w, bias, prev = _inputs(B, Cin, Cout, L, 7, gen, wscale=2.0)
        x, w, bias, prev = x.to(DEV), w.to(DEV), bias.to(DEV), prev[:, :, :L].contiguous().to(DEV)
        xn, pn, xz = x.clone(), prev.clone(), x.clone()
        for b, n in enumerate(clamp):          # never read: NaN in the kernel's input, 0 in the reference's
            xn[b, :, n:] = float("nan")
            pn[b, :, n:] = float("nan")
            xz[b, :, n:] = 0.0
        got, rec = _run_direct(ops, xn, w, bias, 1, 3, flags, pn, xo, 0, 0, valid_len=vl)
        assert (KERNELS[rec["kernel"]], rec["flags"], rec["has_valid_len"]) == (kernel, flags, 1), rec
        assert (rec["grid_x"], rec["grid_y"]) == (-(-L // 512), B), rec
        ref, tol = conv_ref(xz, w, bias, 1, 3, flags, prev)
        for b, n in enumerate(clamp):
            worst = max(worst, _check(got[b, :, :n], ref[b, :, :n], tol[b, :, :n], (kernel, flag_name(flags), b, n)))
            assert bool((got[b, :, n:] == 0).all()), (kernel, flag_name(flags), b, n)
    print(f"\n[parity] direct {kernel} ragged L={L}: 16 flag sets x {B} items, worst error / bound {worst:.3f}")


RAGGED_KEYS = {_key(kn, f, True) for kn in ("thin_vec", "thin_smem") for f in FLAG_SETS}


# ----------------------------------------------------------------------------------------------
# (d) the direct ConvTranspose
# ----------------------------------------------------------------------------------------------
def _convt_pairs():
    """Every (k, u) with u <= 8 the C-ABI accepts: k >= u, k <= 16, <= 4 taps per phase, L_out = u L_in."""
    return [(k, u) for u in range(1, 9) for k in range(u, 17) if -(-k // u) <= 4 and k - 2 * ((k - u) // 2) == u]


CONVT_CIN, CONVT_COUT, CONVT_LIN = (1, 7, 9, 17), (1, 31, 33), (1, 63, 64, 65)


def convt_ref(x, w, bias, u, add):
    """float64 ConvTranspose1d(k, u, padding (k - u) / 2) + add, and its bound (n = Cin x taps per phase + 1)."""
    Cin, k = w.shape[0], w.shape[2]
    p = (k - u) // 2
    x64, w64 = x.double(), w.double()
    y = F.conv_transpose1d(x64, w64, bias.double(), stride=u, padding=p)
    S = F.conv_transpose1d(x64.abs(), w64.abs(), None, stride=u, padding=p)
    n = Cin * -(-k // u) + 1
    tol = LAMBDA * math.sqrt(n) * U32 * (S + bias.double().abs()[None, :, None])
    if add is not None:
        y = y + add.double()
        tol = tol + U32 * y.abs()
    return y, tol


@pytest.mark.gpu
@pytest.mark.parametrize("u", range(1, 9))
def test_conv_transpose_direct_vs_fp64(hsv, u):
    ops = hsv.ops
    pairs = [p for p in _convt_pairs() if p[1] == u]
    worst, seen = 0.0, set()
    for k, _ in pairs:
        for i in range(len(CONVT_CIN) * len(CONVT_LIN)):          # every Cin with every Lin, Cout and add rotating
            Cin, Lin = CONVT_CIN[i % 4], CONVT_LIN[i // 4]
            Cout, with_add = CONVT_COUT[(i + k) % 3], (i + k) % 2 == 1
            B = 2
            gen = torch.Generator().manual_seed(1000 * k + 10 * u + i)
            x = (torch.randn(B, Cin, Lin, generator=gen) * 2).to(DEV)
            w = (torch.randn(Cin, Cout, k, generator=gen) / math.sqrt(Cin)).to(DEV)
            bias = torch.randn(Cout, generator=gen).to(DEV)
            add = torch.randn(B, Cout, u * Lin, generator=gen).to(DEV) if with_add else None
            before = ops.last_launch_config(ops.LAUNCH_DIRECT)["launches"]
            got = ops.conv_transpose1d(x, w, bias, u, add=add)
            rec = ops.last_launch_config(ops.LAUNCH_DIRECT)
            assert rec["launches"] == before + 1
            assert (rec["kernel"], rec["flags"], rec["has_valid_len"]) == (6, ADD if with_add else 0, 0), rec
            assert (rec["grid_x"], rec["grid_y"], rec["grid_z"]) == (-(-Lin // 64), -(-Cout // 32) * u, B), rec
            seen.add(direct_key(rec))
            ref, tol = convt_ref(x, w, bias, u, add)
            worst = max(worst, _check(got, ref, tol, (k, u, Cin, Cout, Lin, with_add)))
    assert seen == {_key("convT", 0), _key("convT", ADD)}, seen
    print(f"\n[parity] direct convT u={u}: k {[p[0] for p in pairs]}, worst error / bound {worst:.3f}")


def test_convt_pairs_include_the_models():
    """The vocoder's (8, 4), (11, 5), (4, 2), SpeechSR's (3, 3) and the edge pairs are among the (k, u) of (d)."""
    pairs = set(_convt_pairs())
    assert {(8, 4), (11, 5), (4, 2), (3, 3), (16, 8), (13, 5), (3, 1), (1, 1)} <= pairs
    assert (2, 1) not in pairs and (5, 1) not in pairs and (9, 2) not in pairs


# ----------------------------------------------------------------------------------------------
# (e) the single-path kernels
# ----------------------------------------------------------------------------------------------
def _sr_ref(ops, x, w, bias, Li, Lo, t0, t1):
    """float64 conv_pre (Cin 1, k 7, pad 3) of x[:Li] at the kernel's own (i0, i1, lam) for outputs [t0, t1), and the
    bound: each conv value within LAMBDA sqrt(8) u (S + |b|), the lerp's fp32 1 - lam, product and fma 3 u of
    |(1 - lam) va| + |lam vb|.  Returns (ref, tol) [C, t1 - t0]."""
    i0, i1, lam = (t[t0:t1] for t in ops.interp_linear_table(Li, Lo, DEV))
    xp = F.pad(x[:Li].double(), (3, 3))
    w64, b64 = w.double()[:, 0], bias.double()[:, None]
    win = lambda i: xp[i.long()[:, None] + torch.arange(7, device=DEV)]          # [T, 7] = x[i - 3 .. i + 3]
    va, vb = win(i0) @ w64.T, win(i1) @ w64.T                                    # [T, C]
    sa, sb = win(i0).abs() @ w64.abs().T, win(i1).abs() @ w64.abs().T
    va, vb, sa, sb = va.T + b64, vb.T + b64, sa.T + b64.abs(), sb.T + b64.abs()
    l64 = lam.double()[None, :]
    ref = (1 - l64) * va + l64 * vb
    e = LAMBDA * math.sqrt(8) * U32
    tol = (1 - l64) * e * sa + l64 * e * sb + 3 * U32 * ((1 - l64) * va.abs() + l64 * vb.abs())
    return ref, tol


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [1.5, 3])
def test_sr_pre_interp_vs_fp64(hsv, scale):
    ops = hsv.ops
    C, worst = 32, 0.0
    gen = torch.Generator().manual_seed(int(scale * 2))
    w = (torch.randn(C, 1, 7, generator=gen) * 0.4).to(DEV)
    bias = torch.randn(C, generator=gen).to(DEV)
    # full: small sizes, and 16 kHz -> 48 kHz on windows at both ends and across the middle
    for Lin in (1, 7, 100, 1001) + ((160000,) if scale == 3 else (48000,)):
        Lout = int(Lin * scale)
        x = (torch.randn(2, 1, Lin, generator=gen) * 0.5).to(DEV)
        got = ops.sr_pre_interp(x, w, bias, Lout)
        wins = [(0, min(Lout, 2048)), (max(0, Lout - 2048), Lout), (max(0, Lout // 2 - 1000), min(Lout, Lout // 2 + 1000))]
        for b in range(2):
            for t0, t1 in wins:
                if t1 <= t0:
                    continue
                ref, tol = _sr_ref(ops, x[b, 0], w, bias, Lin, Lout, t0, t1)
                worst = max(worst, _check(got[b, :, t0:t1], ref, tol, ("full", Lin, b, t0)))
    # ragged: each item interpolated from its own Li to Lo = int(Li * scale); NaN past Li, 0 past Lo
    L = 1001
    lens_in = [L, 0, 1, 7, 500, 999, -3]
    B = len(lens_in)
    Lout = int(L * scale)
    lens_out = [int(max(n, 0) * scale) for n in lens_in]
    x = (torch.randn(B, 1, L, generator=gen) * 0.5).to(DEV)
    for b, n in enumerate(lens_in):
        x[b, :, max(n, 0):] = float("nan")
    vin = torch.tensor(lens_in, dtype=torch.int32, device=DEV)
    vout = torch.tensor(lens_out, dtype=torch.int32, device=DEV)
    got = ops.sr_pre_interp(x, w, bias, Lout, valid_len=(vin, vout))
    for b, (n, m) in enumerate(zip(lens_in, lens_out)):
        if m:
            ref, tol = _sr_ref(ops, x[b, 0], w, bias, n, m, 0, m)
            worst = max(worst, _check(got[b, :, :m], ref, tol, ("ragged", n, m)))
        assert bool((got[b, :, m:] == 0).all()), (b, n, m)
    print(f"\n[parity] sr_pre_interp x{scale}: worst error / bound {worst:.3f}")


@pytest.mark.gpu
@pytest.mark.parametrize("k,stride,pad,Lin", [(9, 4, 4, 4003), (9, 4, 4, 4001), (5, 3, 2, 302), (3, 2, 0, 77)])
def test_conv1d_c1_strided_vs_fp64(hsv, k, stride, pad, Lin):
    """PosteriorSFEncoder.pre_filter's conv (Cin 1, stride 4, pad 4) and other strides, Lin not a multiple of the
    stride; with and without a mask, full and ragged (NaN past stride * valid_len, outputs there exactly 0)."""
    ops = hsv.ops
    B, Cout = 5, 192
    gen = torch.Generator().manual_seed(Lin + k)
    x = (torch.randn(B, 1, Lin, generator=gen) * 3).to(DEV)
    w = (torch.randn(Cout, 1, k, generator=gen) / math.sqrt(k)).to(DEV)
    bias = torch.randn(Cout, generator=gen).to(DEV)
    Lout = (Lin + 2 * pad - k) // stride + 1
    keep = torch.tensor([Lout, Lout - 5, 1, Lout // 2, Lout])
    mask = (torch.arange(Lout)[None, :] < keep[:, None]).float()[:, None, :].to(DEV)

    def ref_of(xx):
        y = F.conv1d(xx.double(), w.double(), bias.double(), stride=stride, padding=pad)
        S = F.conv1d(xx.double().abs(), w.double().abs(), bias.double().abs(), stride=stride, padding=pad)
        return y, LAMBDA * math.sqrt(k + 1) * U32 * S

    worst = 0.0
    for m in (None, mask):
        got = ops.conv1d_c1_strided(x, w, bias, stride, pad, m)
        ref, tol = ref_of(x)
        if m is not None:
            ref = ref * m.double()
        worst = max(worst, _check(got, ref, tol, ("full", m is not None)))
    # ragged: item b is its first nv output frames and min(stride * nv, Lin) input samples
    vlen = [Lout, 0, Lout // 3 + 1, Lout + 9, -2]
    nvs = [min(max(v, 0), Lout) for v in vlen]
    xn, xz = x.clone(), x.clone()
    for b, nv in enumerate(nvs):
        xn[b, :, min(stride * nv, Lin):] = float("nan")
        xz[b, :, min(stride * nv, Lin):] = 0.0
    got = ops.conv1d_c1_strided(xn, w, bias, stride, pad, mask, valid_len=torch.tensor(vlen, dtype=torch.int32,
                                                                                          device=DEV))
    ref, tol = ref_of(xz)
    ref = ref * mask.double()
    for b, nv in enumerate(nvs):
        worst = max(worst, _check(got[b, :, :nv], ref[b, :, :nv], tol[b, :, :nv], ("ragged", b, nv)))
        assert bool((got[b, :, nv:] == 0).all()), (b, nv)
    print(f"\n[parity] conv1d_c1_strided k{k} s{stride} p{pad} Lin={Lin}: worst error / bound {worst:.3f}")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(32, 1, 7), (16, 16, 3), (512, 192, 7), (256, 128, 11), (192, 1024, 7),
                                   (64, 1024, 1), (3, 1, 1), (5, 257, 3)])
def test_weight_norm_fold_vs_fp64(hsv, shape):
    """w = v g / ||v|| at the path's widest rows (inner up to 1024 x 7).  One CTA per row of 256 threads: each thread
    sums its ceil(inner / 256) squares as an fmaf chain, then two 5-level shuffle trees over 32 partials: at most
    d = ceil(inner / 256) + 10 rounded additions of positive terms, so |s - ||v||^2| <= d u ||v||^2 (to first order).
    sqrtf halves that and rounds (0.5 u), g / sqrt and v * sc round once each: |w - w64| <= (d / 2 + 1.5) u |w64|,
    and 2 u more for the second-order terms."""
    gen = torch.Generator().manual_seed(sum(shape))
    v = torch.randn(shape, generator=gen) * 0.05
    v[0] *= 1e3                                          # rows of very different norms
    g = torch.rand(shape[0], 1, 1, generator=gen) + 0.5
    g[-1] = -g[-1]
    w = hsv.ops.weight_norm_fold(v.to(DEV), g.to(DEV)).double().cpu()
    v64 = v.double()
    ref = v64 * (g.double() / v64.flatten(1).norm(dim=1).view(-1, *([1] * (v.dim() - 1))))
    inner = v[0].numel()
    d = -(-inner // 256) + 10
    tol = (d / 2 + 3.5) * U32 * ref.abs()
    r = _check(w, ref, tol, shape)
    print(f"\n[parity] weight_norm_fold {shape}: worst error / bound {r:.3f}")


# ----------------------------------------------------------------------------------------------
# (f) production conv_post shapes, spot-checked on windows
# ----------------------------------------------------------------------------------------------
# (B, Cin, L, flags, kernel): vocoder B = 16 x 10 s, SpeechSR48 B = 16 x 10 s, SpeechSR24 x 10 s, the PitchPredictor
PRODUCTION = [(16, 16, 160000, TANH, "thin_vec"), (16, 32, 480000, TANH, "thin_vec"), (1, 32, 240000, TANH, "thin_vec"),
              (16, 64, 4000, LRELU001, "thin_vec")]


def _windows(L, seed, n=6):
    rng = np.random.default_rng(seed)
    w = [(0, min(L, 1024)), (max(0, L - 1024), L)]
    for s in rng.integers(1, max(2, L // 512 - 1), n):
        w.append((int(s) * 512 - 300, min(L, int(s) * 512 + 300)))
    return w


@pytest.mark.gpu
@pytest.mark.parametrize("B,Cin,L,flags,kernel", PRODUCTION)
def test_production_conv_post_windows_vs_fp64(hsv, B, Cin, L, flags, kernel):
    ops = hsv.ops
    gen = torch.Generator(device=DEV).manual_seed(L + Cin)
    x = torch.randn(B, Cin, L, generator=gen, device=DEV) * 2
    w = torch.randn(1, Cin, 7, generator=gen, device=DEV) * (2 / math.sqrt(Cin * 7))
    got = ops.conv1d_direct(x, w, None, pad=3, flags=flags)
    rec = ops.last_launch_config(ops.LAUNCH_DIRECT)
    assert direct_key(rec) == _key(kernel, flags), rec
    worst = 0.0
    for s, e in _windows(L, L):
        a, z = max(0, s - 3), min(L, e + 3)
        xw = F.pad(x[:, :, a:z], (3 - (s - a), 3 - (z - e)))
        ref, tol = conv_ref(xw, w, None, 1, 0, flags)
        worst = max(worst, _check(got[:, :, s:e], ref, tol, (s, e)))
    print(f"\n[parity] direct conv_post [{B}, {Cin}, {L}] {flag_name(flags)}: worst error / bound {worst:.3f}")


# ----------------------------------------------------------------------------------------------
# (g) census
# ----------------------------------------------------------------------------------------------
VERIFIED = frozenset({_key(kn, f) for kn in KERNEL_SHAPES for f in FLAG_SETS} | RAGGED_KEYS
                     | {_key("convT", 0), _key("convT", ADD)})


def test_verified_covers_every_kernel():
    """Every kernel id 0-6 of the record appears in VERIFIED, and each edge case of (b) runs a verified key."""
    assert {k.split(":")[1] for k in VERIFIED} == set(KERNELS)
    assert {c[0] for c in EDGE_CASES} == set(KERNELS) - {"convT"}


def test_empty_calls_launch_nothing():
    """B = 0, Lout <= 0 and Lin = 0 return before any launch and leave the record unchanged (host-only, no GPU)."""
    from megatts2_hierspeechpp_b200 import _lib, build, ops
    build.build()
    lib = _lib.load()
    before = ops.last_launch_config(ops.LAUNCH_DIRECT)
    assert lib.hsv_conv1d_direct(None, None, None, None, 0, 4, 4, 10, 10, 3, 1, 1, 0, None) == 0
    assert lib.hsv_conv1d_direct(None, None, None, None, 2, 4, 4, 3, -3, 7, 1, 0, 0, None) == 0
    assert lib.hsv_conv1d_direct_ragged(None, None, None, None, None, 0, 4, 1, 10, 10, 7, 1, 3, 0, None) == 0
    assert lib.hsv_conv_transpose1d_direct(None, None, None, None, None, 2, 4, 4, 0, 8, 4, None) == 0
    assert lib.hsv_conv_transpose1d_direct(None, None, None, None, None, 0, 4, 4, 10, 8, 4, None) == 0
    assert ops.last_launch_config(ops.LAUNCH_DIRECT) == before


_DIRECT_CALLS = {"hsv_conv1d_direct", "hsv_conv1d_direct_ragged", "hsv_conv_transpose1d_direct"}


def _record_direct(hsv, monkeypatch, run):
    from megatts2_hierspeechpp_b200 import _lib
    ops = hsv.ops
    seen, orig = {}, _lib.check
    last = [ops.last_launch_config(ops.LAUNCH_DIRECT)["launches"]]

    def recording_check(rc, what):
        orig(rc, what)
        if what in _DIRECT_CALLS:
            c = ops.last_launch_config(ops.LAUNCH_DIRECT)
            if c["launches"] != last[0]:            # B == 0 / Lout <= 0 calls launch nothing
                last[0] = c["launches"]
                k = direct_key(c)
                seen[k] = seen.get(k, 0) + 1

    monkeypatch.setattr(_lib, "check", recording_check)
    try:
        with torch.no_grad():
            run()
        torch.cuda.synchronize()
    finally:
        monkeypatch.setattr(_lib, "check", orig)
    return seen


def _assert_census(name, seen):
    print(f"\n[census] {name} direct: " + ", ".join(f"{k} x{n}" for k, n in sorted(seen.items())))
    assert seen, f"{name}: no CUDA-core conv launch recorded"
    unverified = sorted(set(seen) - VERIFIED)
    assert not unverified, f"{name} launches CUDA-core conv variants no case verifies: {unverified}"


CENSUS = [("vocoder", 1, 10.0), ("vocoder", 16, 10.0), ("speechsr48", 16, 10.0), ("synth", 1, 10.0),
          ("tts", 1, 10.0), ("speechsr24", 1, 10.0), ("chain24", 1, 10.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("workload,batch,seconds", CENSUS, ids=[f"{w}-B{b}" for w, b, _ in CENSUS])
def test_census_workload_direct_verified(hsv, monkeypatch, workload, batch, seconds):
    """One eager forward of a benchmark workload (bench.py's model and inputs)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    import bench

    wl = bench.make_workload(argparse.Namespace(workload=workload, batch=batch, seconds=seconds), 0)
    model = bench.build_model(wl, DEV)
    seen = _record_direct(hsv, monkeypatch, lambda: model(*[t.to(DEV) for t in wl["host_inputs"]]))
    _assert_census(wl["name"], seen)


def _lens(lens):
    return torch.tensor(lens, dtype=torch.int32, device=DEV)


@pytest.mark.gpu
def test_census_ragged_vocoder_and_speechsr48_verified(hsv, monkeypatch):
    from conftest import golden_sd
    from oracle import synth
    voc = hsv.Vocoder()
    voc.load_state_dict(synth.vocoder_sd(1234), strict=True)
    voc.to(DEV).eval()
    lens = [500, 1, 2, 37, 499, 250]
    z, g = synth.vocoder_inputs(len(lens), max(lens), seed=21)
    seen = _record_direct(hsv, monkeypatch, lambda: voc(z.to(DEV), g.to(DEV), lengths=_lens(lens)))
    _assert_census(f"ragged vocoder B={len(lens)}", seen)

    sr = hsv.SpeechSR48(100, 40, **hsv.SR_CFG)
    sr.load_state_dict(golden_sd("speechsr48_state.npz"), strict=True)
    sr.to(DEV).eval()
    lens = [48000, 1, 7, 16001, 3333]
    x = torch.randn(len(lens), 1, max(lens), generator=torch.Generator().manual_seed(48)) * 0.3
    seen = _record_direct(hsv, monkeypatch, lambda: sr(x.to(DEV), lengths=_lens(lens)))
    _assert_census(f"ragged SpeechSR48 B={len(lens)}", seen)


@pytest.mark.gpu
def test_census_ragged_ttv_tail_verified(hsv, monkeypatch):
    from oracle import synth
    tail = hsv.TTVTail()
    tail.load_state_dict(synth.ttv_tail_sd(3456), strict=True)
    tail.to(DEV).eval()
    lens = [333, 300, 129, 1, 2]
    z, _, g = synth.ttv_tail_inputs(len(lens), max(lens), seed=22)
    seen = _record_direct(hsv, monkeypatch, lambda: tail(z.to(DEV), None, g.to(DEV), lengths=_lens(lens)))
    _assert_census(f"ragged text-to-vec tail B={len(lens)}", seen)


@pytest.mark.gpu
def test_census_per_item_synthesizer_direct_verified(hsv, monkeypatch):
    """A per-item synthesizer batch of 16 mixed source and prompt lengths, padded as runtime.ragged_prompt_batches
    pads them."""
    from megatts2_hierspeechpp_b200 import synthetic
    from megatts2_hierspeechpp_b200.runtime import ragged_prompt_batches
    from oracle import synth

    model = hsv.HierSpeechSynthesizer()
    model.load_state_dict(synth.synthesizer_sd(1234), strict=True)
    model.to(DEV).eval()
    gen = torch.Generator().manual_seed(16)
    n = 16
    lengths = torch.randint(20, 501, (n,), generator=gen).tolist()
    prompts = torch.randint(20, 301, (n,), generator=gen).tolist()
    ins = [synthetic.synthesizer_inputs(T, Tm, seed=1111 + i) for i, (T, Tm) in enumerate(zip(lengths, prompts))]
    batches = ragged_prompt_batches(range(n), lengths, prompts, n)
    seen = {}
    for ids, Tp, Tmp in batches:
        B = len(ids)
        src, f0 = torch.zeros(B, 1024, Tp), torch.zeros(B, 1, 4 * Tp)
        mel = torch.zeros(2 * B, 80, Tmp)
        for j, i in enumerate(ids):
            T, Tm = lengths[i], prompts[i]
            src[j, :, :T], f0[j, :, :4 * T] = ins[i][0][0], ins[i][1][0]
            mel[j, :, :Tm], mel[B + j, :, :Tm] = ins[i][2][0], ins[i][2][1]
        vl = _lens([lengths[i] for i in ids])
        tl = _lens([prompts[i] for i in ids] * 2)
        s = _record_direct(hsv, monkeypatch, lambda: model.voice_conversion_noise_control(
            src.to(DEV), vl, mel.to(DEV), tl, f0.to(DEV), 0.333, False, 0.3, per_item=True))
        for k, c in s.items():
            seen[k] = seen.get(k, 0) + c
    _assert_census(f"per-item synthesizer B={n} ({len(batches)} batches)", seen)
