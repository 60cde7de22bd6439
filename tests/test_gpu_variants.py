"""Every launch variant of the tcgen05 conv and of the fused activation against a high-precision reference.

The host code of both hot kernels picks an instantiation per launch from the shape: the conv its sub-tiles per CTA
(msub), 4 or 8 warps, the float4 or the scalar / strided epilogue, the one-tile or the persistent kernel (weights in a
ring or resident, one or two A buffers); the activation its run length R.  Small test shapes only ever select the
simplest variants, so every case here forces (a, c) or naturally selects (b) a variant, reads what actually ran through
``ops.last_launch_config`` (the forcing flags are only requests: the host clamps them), and checks the result

* conv: against F.conv1d / F.conv_transpose1d in fp64 on the fp16-rounded operands (bias / residual / addends in fp64),
  2e-4 x max(1, peak), and bit for bit against the msub = 1, default-warp kernel on the same inputs: the MMA K order and
  the epilogue formula (conv + bias) + residual do not depend on the variant;
* activation: against the fp32 oracle (1e-5 x max(1, peak)) and the fp64 closed form, over the whole tensor including
  both replicate-clamped edges, and bit for bit across run lengths (one thread computes an output over the same taps
  whatever R is); the ragged body (valid_len given, a separately inlined copy of the kernel body) at every run length
  with item lengths on both sides of a 16 R-step tile edge, against the fp64 closed form of each item alone.

(d) is a census: the variant of every conv / activation launch of the benchmark workloads must be in ``VERIFIED``, the
set of variants the cases above check (activation keys ``act:R{R}:{f32|blk16}:{full|ragged}``).  A policy change that
ships a new variant fails it until a case covers it.  The SpeechSR24, streaming SpeechSR and ragged-batch entry points
are censused by test_gpu_sr_variants.py.
The operand-writing epilogue's variants (``operand-out:{mode}:n{n_tile}``) are checked against fp64 by
test_gpu_front_variants.py (c), which declares them in ``OPERAND_KEYS``.
"""
import argparse
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import closed_form as CF
from oracle import functional as OF
from test_gpu_front_variants import OPERAND_KEYS, operand_key

DEV = "cuda:0"
SLOT = 11          # blk16 workspace slot of this file (modules use 0..7 and 15, other tests 7..10)

# hsv_set_umma_debug bits (csrc/conv_umma.cu)
RING16, NO_RESIDENT, SCALAR, NARROW, NO_PERSIST, FORCE_PERSIST = 1, 2, 16, 32, 64, 128


def MSUB(m):
    return m << 24


BASE_FLAGS = MSUB(1) | NO_PERSIST   # the reference variant of the bit-identity checks: 128-row tiles, default warps


# ----------------------------------------------------------------------------------------------
# variant keys
# ----------------------------------------------------------------------------------------------
def conv_key(c):
    """Variant key of a conv launch from its ``last_launch_config`` record."""
    kind = c["kind"]
    if kind == 1:
        return f"persist:{'resident' if c['resident'] else 'ring'}:a{c['nabuf']}"
    if kind == 2:
        return "fused-act"
    if kind == 3:
        return operand_key(c["blk_mode"], c["n_tile"])
    if c["nphase"] > 1:
        return f"convT:m{c['msub']}:w{c['warps']}:n{c['n_tile']}"
    return f"conv:m{c['msub']}:w{c['warps']}:{'vec' if c['vec_epi'] else 'scalar'}:n{c['n_tile']}"


def act_key(c):
    if c["mma"]:
        return "act:mma"
    return f"act:R{c['R']}:{'blk16' if c['out_mode'] else 'f32'}:{'ragged' if c['has_valid_len'] else 'full'}"


# ----------------------------------------------------------------------------------------------
# (a) forced conv matrix
# ----------------------------------------------------------------------------------------------
# (cin, cout, k, d, n_tile, L, msub, warps, epilogue); L = 512 m + r puts the ragged last CTA at every sub-tile
# position: r = 1 (one valid row, three empty sub-tiles), 130 (L % 4 = 2), 383 / 384, 4 and 260 (float4: L % 4 = 0)
def _conv_matrix():
    cases = []
    shapes = {16: (48, 32), 32: (192, 64), 64: (48, 128), 128: (128, 256), 256: (64, 256)}
    kd = [(11, 5), (3, 1), (7, 3), (5, 1)]
    l_vec = [4, 260, 384]
    l_sca = [1, 130, 383]
    i = 0
    for nt, (cin, cout) in shapes.items():
        for msub in (1, 2, 4):
            if msub * nt > 512:
                continue
            for warps in ((4, 8) if nt >= 128 and msub < 4 else (4,)):
                for epi in ("vec", "scalar"):
                    k, d = kd[i % len(kd)]
                    r = (l_vec if epi == "vec" else l_sca)[i % 3]
                    L = 512 * (1 + i % 3) + r
                    c = min(cin, 128) if msub == 4 else cin       # msub = 4 with three 64-channel chunks does not fit
                    cases.append((c, cout, k, d, nt, L, msub, warps, epi))
                    i += 1
    return cases


CONV_MATRIX = _conv_matrix()

# ConvTranspose1d (the vocoder's ups[i]: (k, u) = (8, 4), (11, 5), (4, 2)): (cin, cout, k, u, n_tile, Lin, msub, warps)
CONVT_MATRIX = [
    (128, 64, 8, 4, 64, 513, 1, 4), (128, 64, 8, 4, 64, 642, 2, 4), (128, 64, 8, 4, 32, 897, 4, 4),
    (256, 128, 11, 5, 128, 385, 1, 8), (256, 128, 11, 5, 128, 641, 1, 4), (256, 128, 11, 5, 128, 1025, 2, 8),
    (256, 128, 11, 5, 128, 770, 2, 4), (128, 128, 11, 5, 128, 1153, 4, 4),
    (64, 32, 4, 2, 32, 513, 1, 4), (64, 32, 4, 2, 32, 1154, 2, 4), (64, 32, 4, 2, 32, 1409, 4, 4),
    (32, 16, 4, 2, 16, 515, 1, 4), (32, 16, 4, 2, 16, 1030, 2, 4), (32, 16, 4, 2, 16, 2049, 4, 4),
]

# persistent kernel (forced on): (cin/cout, k, d, n_tile, B, L, extra flags, expected key)
PERSIST_MATRIX = [
    (128, 7, 3, 128, 3, 4100, 0, "persist:ring:a2"),
    (128, 11, 5, 128, 2, 2564, RING16, "persist:ring:a2"),
    (256, 11, 5, 128, 2, 3076, 0, "persist:ring:a1"),
    (256, 11, 5, 128, 2, 2052, RING16, "persist:ring:a1"),
    (64, 11, 5, 64, 3, 5124, 0, "persist:resident:a2"),
    (64, 7, 1, 64, 2, 2052, NO_RESIDENT, "persist:ring:a2"),
    (32, 11, 5, 32, 4, 1540, 0, "persist:resident:a2"),
]


def _conv_key_expected(cin, cout, nt, msub, warps, epi, transposed=False):
    if transposed:
        return f"convT:m{msub}:w{warps}:n{nt}"
    return f"conv:m{msub}:w{warps}:{epi}:n{nt}"


def _flags(nt, msub, warps, epi):
    f = MSUB(msub) | NO_PERSIST
    if epi == "scalar":
        f |= SCALAR
    if warps == 4 and nt >= 128:
        f |= NARROW
    return f


# ----------------------------------------------------------------------------------------------
# (c) activation run lengths
# ----------------------------------------------------------------------------------------------
RUNS = (9, 17, 21, 25)


def _act_shapes(R):
    T = 16 * R   # time steps of one CTA tile
    return [(1, 16, 1), (2, 16, 2), (2, 16, T - 1), (1, 32, T), (1, 16, T + 1), (2, 16, 5 * T + 7), (3, 5, 3 * T + 3),
            (1, 7, 2 * T - 2)]


# natural policy: (B, C, L, R the policy picks)
ACT_NATURAL = [(1, 256, 2000, 17), (1, 16, 160000, 21), (16, 32, 80000, 25)]

# natural-policy conv layers at the shapes the workloads run: (name, kind, B, cin, cout, k, d or u, L, expected key)
CONV_NATURAL = [
    ("vocoder ups[3] B=1", "T", 1, 64, 32, 4, 2, 40000, "convT:m1:w4:n32"),
    ("vocoder ups[4] B=1", "T", 1, 32, 16, 4, 2, 80000, "convT:m4:w4:n16"),
    ("vocoder ups[1] B=16", "T", 16, 256, 128, 11, 5, 2000, "convT:m2:w8:n128"),
    ("C=32 dense B=4", "C", 4, 32, 32, 11, 5, 80000, "conv:m4:w4:vec:n32"),
    ("C=64 AMP B=16", "C", 16, 64, 64, 3, 1, 40000, "persist:resident:a2"),
    ("C=128 AMP B=16", "C", 16, 128, 128, 7, 3, 10000, "persist:ring:a2"),
    ("C=256 AMP B=16", "C", 16, 256, 256, 11, 5, 2000, "persist:ring:a1"),
    ("SpeechSR48 C=32 odd L", "C", 1, 32, 32, 11, 5, 480001, "conv:m4:w4:scalar:n32"),
]

# ----------------------------------------------------------------------------------------------
# (d) the variants (a)-(c) verify, and the operand-writing epilogue's (test_gpu_front_variants.py (c)).  "fused-act"
# (hsv_act_conv1d_umma) is checked by test_gpu_kernels.py::test_act_conv_fused_equals_unfused; it is listed here on the
# strength of that test.
# ----------------------------------------------------------------------------------------------
VERIFIED = set(OPERAND_KEYS) | {
    "fused-act",
    "persist:ring:a2", "persist:ring:a1", "persist:resident:a2",
    "conv:m1:w4:vec:n16", "conv:m1:w4:scalar:n16", "conv:m2:w4:vec:n16", "conv:m2:w4:scalar:n16",
    "conv:m4:w4:vec:n16", "conv:m4:w4:scalar:n16",
    "conv:m1:w4:vec:n32", "conv:m1:w4:scalar:n32", "conv:m2:w4:vec:n32", "conv:m2:w4:scalar:n32",
    "conv:m4:w4:vec:n32", "conv:m4:w4:scalar:n32",
    "conv:m1:w4:vec:n64", "conv:m1:w4:scalar:n64", "conv:m2:w4:vec:n64", "conv:m2:w4:scalar:n64",
    "conv:m4:w4:vec:n64", "conv:m4:w4:scalar:n64",
    "conv:m1:w4:vec:n128", "conv:m1:w4:scalar:n128", "conv:m1:w8:vec:n128", "conv:m1:w8:scalar:n128",
    "conv:m2:w4:vec:n128", "conv:m2:w4:scalar:n128", "conv:m2:w8:vec:n128", "conv:m2:w8:scalar:n128",
    "conv:m4:w4:vec:n128", "conv:m4:w4:scalar:n128",
    "conv:m1:w4:vec:n256", "conv:m1:w4:scalar:n256", "conv:m1:w8:vec:n256", "conv:m1:w8:scalar:n256",
    "conv:m2:w4:vec:n256", "conv:m2:w4:scalar:n256", "conv:m2:w8:vec:n256", "conv:m2:w8:scalar:n256",
    "convT:m1:w4:n64", "convT:m2:w4:n64", "convT:m4:w4:n32",
    "convT:m1:w8:n128", "convT:m1:w4:n128", "convT:m2:w8:n128", "convT:m2:w4:n128", "convT:m4:w4:n128",
    "convT:m1:w4:n32", "convT:m2:w4:n32", "convT:m1:w4:n16", "convT:m2:w4:n16", "convT:m4:w4:n16",
}
VERIFIED |= {f"act:R{R}:{m}:{form}" for R in RUNS for m in ("f32", "blk16") for form in ("full", "ragged")}


def _declared_keys():
    """The variant keys the cases of (a)-(c) assert (each case checks its key through the hook when it runs)."""
    keys = {"fused-act"} | set(OPERAND_KEYS)
    keys |= {_conv_key_expected(c[0], c[1], c[4], c[6], c[7], c[8]) for c in CONV_MATRIX}
    keys |= {_conv_key_expected(c[0], c[1], c[4], c[6], c[7], None, True) for c in CONVT_MATRIX}
    keys |= {c[-1] for c in PERSIST_MATRIX}
    keys |= {c[-1] for c in CONV_NATURAL}
    keys |= {f"act:R{R}:{m}:full" for R in RUNS for m in ("f32", "blk16")}
    keys |= {f"act:R{R}:{m}:ragged" for R in RUNS for m in ("f32", "blk16")}
    return keys


def test_verified_set_is_covered_by_the_cases():
    """Every key in VERIFIED is asserted by a case of this file (no GPU needed: the cases declare their keys)."""
    missing = VERIFIED - _declared_keys()
    assert not missing, sorted(missing)


def test_last_launch_config_hook_four_families_ragged_act():
    """The hook reports the documented fields of its four families (conv, activation with its valid_len flag,
    attention, CUDA-core conv) and rejects an unknown family (host-only, no GPU)."""
    from megatts2_hierspeechpp_b200 import _lib, build, ops
    build.build()
    assert set(ops.last_launch_config(ops.LAUNCH_CONV)) >= {"kind", "msub", "warps", "vec_epi", "blk_mode", "launches"}
    assert tuple(ops.last_launch_config(ops.LAUNCH_ACT)) == ("R", "mma", "out_mode", "has_valid_len", "launches")
    assert _lib.load().hsv_last_launch_config(1, None, 0) == 5
    assert set(ops.last_launch_config(ops.LAUNCH_MHA)) >= {"kernel", "D", "out_mode", "kv16", "q16", "launches"}
    assert tuple(ops.last_launch_config(ops.LAUNCH_DIRECT)) == ("kernel", "flags", "has_valid_len", "grid_x", "grid_y",
                                                                "grid_z", "launches")
    assert _lib.load().hsv_last_launch_config(3, None, 0) == 7
    assert _lib.load().hsv_last_launch_config(4, None, 0) < 0
    assert _lib.load().hsv_last_launch_config(-1, None, 0) < 0


# ----------------------------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------------------------
def _tol(ref):
    return 2e-4 * max(1.0, ref.abs().max().item())


class _Flags:
    """hsv_set_umma_debug / hsv_set_act_variant for a block, restored to 0 on the way out."""

    def __init__(self, ops, umma=None, act=None):
        self.ops, self.umma, self.act = ops, umma, act

    def __enter__(self):
        if self.umma is not None:
            self.ops.set_umma_debug(self.umma)
        if self.act is not None:
            self.ops.set_act_variant(self.act)

    def __exit__(self, *exc):
        self.ops.set_umma_debug(0)
        self.ops.set_act_variant(0)


def _conv_data(B, cin, cout, k, Lout, seed, u=None):
    gen = torch.Generator().manual_seed(seed)
    Lin = Lout if u is None else Lout // u
    x = torch.randn(B, cin, Lin, generator=gen)
    if u is None:
        w = torch.randn(cout, cin, k, generator=gen) / (cin * k) ** 0.5
    else:
        w = torch.randn(cin, cout, k, generator=gen) / (cin * k / u) ** 0.5
    b = torch.randn(cout, generator=gen) * 0.1
    res = torch.randn(B, cout, Lout, generator=gen)
    return x.to(DEV), w.to(DEV), b.to(DEV), res.to(DEV)


def _ref_conv(x, w, b, k, d):
    """fp64 reference on the kernel's fp16-rounded operands (on the GPU: the natural-policy shapes are large)."""
    return F.conv1d(x.half().double(), w.half().double(), None if b is None else b.double(),
                    padding=OF.get_padding(k, d), dilation=d)


def _ref_convT(x, w, b, k, u):
    return F.conv_transpose1d(x.half().double(), w.half().double(), None if b is None else b.double(), stride=u,
                              padding=(k - u) // 2)


def _conv_outputs(ops, buf, wp, b, res, L, cin, cout, k, d, nt):
    """One launch per output mode; returns {mode: tensor} and the variant key of every launch."""
    keys, outs = set(), {}

    def run(**kw):
        y = ops.conv1d_umma(buf, wp, kw.pop("bias", b), L, cin, cout, k, d, nt, **kw)
        keys.add(conv_key(ops.last_launch_config(ops.LAUNCH_CONV)))
        return y

    outs["res"] = run(residual=res)
    r2 = res.clone()
    run(residual=r2, out=r2)                     # out aliasing residual: the AMP block's in-place update
    outs["inplace"] = r2
    acc = torch.full_like(res, float("nan"))
    for mode in (ops.ACC_SET, ops.ACC_ADD, ops.ACC_ADD):
        run(acc=acc, acc_mode=mode, want_out=False)
    outs["acc3"] = acc
    outs["nobias"] = run(bias=None)
    return outs, keys


def _check_conv_modes(outs, ref_nb, b, res):
    ref = ref_nb + b.double().view(1, -1, 1)
    want = {"res": ref + res.double(), "inplace": ref + res.double(), "acc3": 3 * ref, "nobias": ref_nb}
    for m, y in outs.items():
        err = (y.double() - want[m]).abs().max().item()
        assert err <= _tol(want[m]), (m, err)


# ----------------------------------------------------------------------------------------------
# (a) forced conv matrix
# ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cin,cout,k,d,nt,L,msub,warps,epi", CONV_MATRIX)
def test_conv_forced_variant(hsv, cin, cout, k, d, nt, L, msub, warps, epi):
    ops = hsv.ops
    B = 2
    x, w, b, res = _conv_data(B, cin, cout, k, L, seed=cin + 7 * nt + L + 13 * msub + warps)
    buf = ops.blk16_buffer(B, cin, L, DEV, slot=SLOT)
    ops.pack_blk16(x, buf)
    wp = ops.pack_conv_weight(w, nt)
    want_key = _conv_key_expected(cin, cout, nt, msub, warps, epi)
    try:
        with _Flags(ops, umma=_flags(nt, msub, warps, epi)):
            outs, keys = _conv_outputs(ops, buf, wp, b, res, L, cin, cout, k, d, nt)
        with _Flags(ops, umma=BASE_FLAGS):
            base, _ = _conv_outputs(ops, buf, wp, b, res, L, cin, cout, k, d, nt)
    finally:
        ops.set_umma_debug(0)
    assert keys == {want_key}, (keys, want_key)
    _check_conv_modes(outs, _ref_conv(x, w, None, k, d), b, res)
    for m in outs:
        assert torch.equal(outs[m], base[m]), (m, (outs[m] - base[m]).abs().max().item())


@pytest.mark.gpu
@pytest.mark.parametrize("cin,cout,k,u,nt,Lin,msub,warps", CONVT_MATRIX)
def test_convT_forced_variant(hsv, cin, cout, k, u, nt, Lin, msub, warps):
    ops = hsv.ops
    B = 2
    x, w, b, add = _conv_data(B, cin, cout, k, u * Lin, seed=cin + k + Lin + msub, u=u)
    buf = ops.blk16_buffer(B, cin, Lin, DEV, slot=SLOT)
    ops.pack_blk16(x, buf)
    wp = ops.pack_convT_weight(w, u, nt)
    want_key = _conv_key_expected(cin, cout, nt, msub, warps, None, True)
    outs, base, keys = {}, {}, set()
    try:
        for flags, dst in ((_flags(nt, msub, warps, "scalar"), outs), (BASE_FLAGS, base)):
            with _Flags(ops, umma=flags):
                dst["add"] = ops.conv_transpose1d_umma(buf, wp, b, Lin, cin, cout, k, u, nt, add=add)
                if dst is outs:
                    keys.add(conv_key(ops.last_launch_config(ops.LAUNCH_CONV)))
                dst["nobias"] = ops.conv_transpose1d_umma(buf, wp, None, Lin, cin, cout, k, u, nt)
                if dst is outs:
                    keys.add(conv_key(ops.last_launch_config(ops.LAUNCH_CONV)))
    finally:
        ops.set_umma_debug(0)
    assert keys == {want_key}, (keys, want_key)
    ref_nb = _ref_convT(x, w, None, k, u)
    want = {"add": ref_nb + b.double().view(1, -1, 1) + add.double(), "nobias": ref_nb}
    for m in outs:
        err = (outs[m].double() - want[m]).abs().max().item()
        assert err <= _tol(want[m]), (m, err)
        assert torch.equal(outs[m], base[m]), (m, (outs[m] - base[m]).abs().max().item())


@pytest.mark.gpu
@pytest.mark.parametrize("C,k,d,nt,B,L,extra,want_key", PERSIST_MATRIX)
def test_conv_persistent_variant_vs_fp64(hsv, C, k, d, nt, B, L, extra, want_key):
    ops = hsv.ops
    x, w, b, res = _conv_data(B, C, C, k, L, seed=C + k + L + extra)
    buf = ops.blk16_buffer(B, C, L, DEV, slot=SLOT)
    ops.pack_blk16(x, buf)
    wp = ops.pack_conv_weight(w, nt)
    try:
        with _Flags(ops, umma=FORCE_PERSIST | extra):
            outs, keys = _conv_outputs(ops, buf, wp, b, res, L, C, C, k, d, nt)
        with _Flags(ops, umma=BASE_FLAGS):
            base, _ = _conv_outputs(ops, buf, wp, b, res, L, C, C, k, d, nt)
    finally:
        ops.set_umma_debug(0)
    assert keys == {want_key}, (keys, want_key)
    _check_conv_modes(outs, _ref_conv(x, w, None, k, d), b, res)
    for m in outs:
        assert torch.equal(outs[m], base[m]), (m, (outs[m] - base[m]).abs().max().item())


# ----------------------------------------------------------------------------------------------
# (b) natural policy at the production layer shapes
# ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name,kind,B,cin,cout,k,du,L,want_key", CONV_NATURAL, ids=[c[0] for c in CONV_NATURAL])
def test_conv_natural_policy(hsv, name, kind, B, cin, cout, k, du, L, want_key):
    ops = hsv.ops
    ops.set_umma_debug(0)
    row_tiles = B * ((L + ops.TILE_M - 1) // ops.TILE_M)
    if kind == "T":
        x, w, b, add = _conv_data(B, cin, cout, k, du * L, seed=L + cin, u=du)
        buf = ops.blk16_buffer(B, cin, L, DEV, slot=SLOT)
        ops.pack_blk16(x, buf)
        nt = ops.pick_n_tile(cout, row_tiles * du)             # modules._Folded.packedT_weight
        y = ops.conv_transpose1d_umma(buf, ops.pack_convT_weight(w, du, nt), b, L, cin, cout, k, du, nt, add=add)
        key = conv_key(ops.last_launch_config(ops.LAUNCH_CONV))
        ref = _ref_convT(x, w, b, k, du) + add.double()
    else:
        x, w, b, res = _conv_data(B, cin, cout, k, L, seed=L + cin)
        buf = ops.blk16_buffer(B, cin, L, DEV, slot=SLOT)
        ops.pack_blk16(x, buf)
        nt = ops.pick_n_tile(cout, row_tiles, cin * k)        # modules._Folded.packed_weight
        y = ops.conv1d_umma(buf, ops.pack_conv_weight(w, nt), b, L, cin, cout, k, du, nt, residual=res)
        key = conv_key(ops.last_launch_config(ops.LAUNCH_CONV))
        ref = _ref_conv(x, w, b, k, du) + res.double()
    assert key == want_key, (name, key)
    err = (y.double() - ref).abs()
    assert err.max().item() <= _tol(ref), (name, err.max().item(), divmod(int(err.argmax()) % y.shape[-1], 512))


# ----------------------------------------------------------------------------------------------
# (c) activation run lengths
# ----------------------------------------------------------------------------------------------
def _act_params(C, seed):
    gen = torch.Generator().manual_seed(seed)
    al = torch.rand(C, generator=gen) * 1.5 - 0.5      # checkpoint-range log-scale alpha / beta
    be = torch.rand(C, generator=gen) * 1.3 - 0.5
    return al, be


def _act_oracle(x, al, be):
    taps = torch.from_numpy(CF.FILTER_TAPS_F32.copy()).view(1, 1, 12)
    sd = {"a.act.alpha": al, "a.act.beta": be, "a.upsample.filter": taps, "a.downsample.lowpass.filter": taps}
    return OF.activation1d(sd, "a.", x)


def _fp16_neighbour_ok(y, ref):
    """The fp16 operand holds the fp32 result rounded to fp16: within one fp16 spacing of the reference (plus the fp32
    tolerance, which decides the rounding direction only near a midpoint)."""
    a = ref.abs()
    ulp = torch.exp2(torch.floor(torch.log2(a.clamp_min(2.0 ** -14))) - 10)
    return bool(((y - ref).abs() <= ulp + 1e-5 * max(1.0, a.max().item())).all())


def _act_run(ops, x, al, be, R, blk, valid_len=None):
    """The activation forced to run length R; returns (fp32 [B,C,L] result, key that ran)."""
    B, C, L = x.shape
    try:
        with _Flags(ops, act=R << 8):
            if blk:
                buf = ops.blk16_buffer(B, C, L, DEV, slot=SLOT)
                ops.act1d_blk16(x, al, be, buf, valid_len=valid_len)
                key = act_key(ops.last_launch_config(ops.LAUNCH_ACT))
                y = ops.unpack_blk16(buf, C, L)
            else:
                y = ops.act1d(x, al, be, valid_len=valid_len)
                key = act_key(ops.last_launch_config(ops.LAUNCH_ACT))
    finally:
        ops.set_act_variant(0)
    return y, key


@pytest.mark.gpu
@pytest.mark.parametrize("blk", [False, True], ids=["f32", "blk16"])
@pytest.mark.parametrize("R", RUNS)
def test_act_run_length_vs_oracle(hsv, R, blk):
    ops = hsv.ops
    for i, (B, C, L) in enumerate(_act_shapes(R)):
        if blk and C % 16:
            continue
        gen = torch.Generator().manual_seed(1000 * R + i)
        x = torch.randn(B, C, L, generator=gen) * 1.5
        al, be = _act_params(C, R + i)
        ref = _act_oracle(x, al, be)
        y, key = _act_run(ops, x.to(DEV), al.to(DEV), be.to(DEV), R, blk)
        assert key == f"act:R{R}:{'blk16' if blk else 'f32'}:full", key
        y = y.cpu()
        if blk:
            assert _fp16_neighbour_ok(y, ref), ((B, C, L), (y - ref).abs().max().item())
        else:
            err = (y - ref).abs()
            assert err.max().item() <= 1e-5 * max(1.0, ref.abs().max().item()), ((B, C, L), err.max().item(),
                                                                                int(err.argmax()) % L)
            if L <= 2000:
                cf = CF.activation1d(x.numpy(), al.numpy(), be.numpy())
                assert np.abs(y.numpy() - cf).max() <= 1e-4 * max(1.0, np.abs(cf).max()), (B, C, L)


@pytest.mark.gpu
def test_act_run_lengths_bit_identical(hsv):
    """Every run length computes every output with the same arithmetic: the four instantiations agree bit for bit."""
    ops = hsv.ops
    gen = torch.Generator().manual_seed(5)
    for (B, C, L) in ((2, 16, 1201), (1, 32, 4096), (3, 16, 401), (1, 16, 7)):
        x = (torch.randn(B, C, L, generator=gen) * 1.5).to(DEV)
        al, be = (t.to(DEV) for t in _act_params(C, L))
        for blk in (False, True):
            ys = [_act_run(ops, x, al, be, R, blk)[0] for R in RUNS]
            for R, y in zip(RUNS[1:], ys[1:]):
                assert torch.equal(y, ys[0]), (B, C, L, R, blk, (y - ys[0]).abs().max().item())


def _ragged_lens(R):
    """(L, valid lengths): 0, 1, both sides of the first 16 R-step tile edge, and the full row."""
    T = 16 * R
    L = 3 * T + 5
    return L, [0, 1, T - 1, T, T + 1, L]


@pytest.mark.gpu
@pytest.mark.parametrize("blk", [False, True], ids=["f32", "blk16"])
@pytest.mark.parametrize("R", RUNS)
def test_act_ragged_run_length_vs_fp64(hsv, R, blk):
    """The ragged body (valid_len given) at every run length: each item against the fp64 closed form on its own
    valid_len[b] steps (the replicate clamp at its length, not at L), NaN past the length never read, exact zeros
    written there, and bit for bit the dense kernel on the item alone."""
    ops = hsv.ops
    L, lens = _ragged_lens(R)
    B, C = len(lens), 32
    gen = torch.Generator().manual_seed(77 * R + blk)
    x = torch.randn(B, C, L, generator=gen) * 1.5
    for b, n in enumerate(lens):
        x[b, :, n:] = float("nan")
    al, be = _act_params(C, R)
    vl = torch.tensor(lens, dtype=torch.int32, device=DEV)
    y, key = _act_run(ops, x.to(DEV), al.to(DEV), be.to(DEV), R, blk, valid_len=vl)
    assert key == f"act:R{R}:{'blk16' if blk else 'f32'}:ragged", key
    for b, n in enumerate(lens):
        assert bool((y[b, :, n:] == 0).all()), (b, n)
        if n == 0:
            continue
        alone, _ = _act_run(ops, x[b:b + 1, :, :n].contiguous().to(DEV), al.to(DEV), be.to(DEV), R, blk)
        assert torch.equal(y[b:b + 1, :, :n], alone), (b, n)
        got = y[b, :, :n].cpu().double().numpy()
        cf = CF.activation1d(x[b:b + 1, :, :n].numpy(), al.numpy(), be.numpy())[0]
        tol = 1e-4 * max(1.0, np.abs(cf).max())
        if blk:
            a = np.abs(cf)
            tol = tol + np.exp2(np.floor(np.log2(np.maximum(a, 2.0 ** -14))) - 10)
        assert (np.abs(got - cf) <= tol).all(), (b, n, np.abs(got - cf).max())


def _windows(L, n, seed):
    """First and last 1024 steps plus n seeded windows straddling 512-step boundaries: [(start, stop)]."""
    rng = np.random.default_rng(seed)
    w = [(0, min(L, 1024)), (max(0, L - 1024), L)]
    for s in rng.integers(1, max(2, L // 512 - 1), n):
        w.append((int(s) * 512 - 300, min(L, int(s) * 512 + 300)))
    return w


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,L,R", ACT_NATURAL)
def test_act_natural_policy(hsv, B, C, L, R):
    ops = hsv.ops
    ops.set_act_variant(0)
    gen = torch.Generator().manual_seed(L + C)
    x = torch.randn(B, C, L, generator=gen) * 1.5
    al, be = _act_params(C, L)
    y = ops.act1d(x.to(DEV), al.to(DEV), be.to(DEV))
    assert act_key(ops.last_launch_config(ops.LAUNCH_ACT)) == f"act:R{R}:f32:full"
    buf = ops.blk16_buffer(B, C, L, DEV, slot=SLOT)
    ops.act1d_blk16(x.to(DEV), al.to(DEV), be.to(DEV), buf)
    assert act_key(ops.last_launch_config(ops.LAUNCH_ACT)) == f"act:R{R}:blk16:full"
    yb = ops.unpack_blk16(buf, C, L).cpu()
    y = y.cpu()
    H = 16   # halo: an output depends on 6 inputs either side
    for s, e in _windows(L, 8, L):
        a, z = max(0, s - H), min(L, e + H)
        ref = _act_oracle(x[:, :, a:z], al, be)[:, :, s - a:e - a]
        err = (y[:, :, s:e] - ref).abs().max().item()
        assert err <= 1e-5 * max(1.0, ref.abs().max().item()), (s, e, err)
        assert _fp16_neighbour_ok(yb[:, :, s:e], ref), (s, e)


# ----------------------------------------------------------------------------------------------
# (d) census of the benchmark workloads
# ----------------------------------------------------------------------------------------------
CENSUS = [("vocoder", 1, 10.0), ("vocoder", 16, 10.0), ("speechsr48", 16, 10.0), ("synth", 1, 10.0), ("tts", 1, 10.0)]
_CONV_CALLS = {"hsv_conv1d_umma", "hsv_conv1d_umma_blk16", "hsv_conv1d_umma_wn_tail", "hsv_act_conv1d_umma",
               "hsv_conv_transpose1d_umma"}


@pytest.mark.gpu
@pytest.mark.parametrize("workload,batch,seconds", CENSUS, ids=[f"{w}-B{b}" for w, b, _ in CENSUS])
def test_census_workload_variants_verified(hsv, monkeypatch, workload, batch, seconds):
    """One eager forward of a benchmark workload (bench.py's model and inputs): the variant of every conv and
    activation launch must be one that (a)-(c) verify."""
    from megatts2_hierspeechpp_b200 import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    import bench

    ops = hsv.ops
    ops.set_umma_debug(0)
    ops.set_act_variant(0)
    seen = {}
    orig = _lib.check

    def recording_check(rc, what):
        orig(rc, what)
        fam = ops.LAUNCH_CONV if what in _CONV_CALLS else (ops.LAUNCH_ACT if what == "hsv_act1d_snakebeta" else None)
        if fam is not None:
            c = ops.last_launch_config(fam)
            if c["launches"] != last[fam]:          # B == 0 / L == 0 calls launch nothing
                last[fam] = c["launches"]
                k = conv_key(c) if fam == ops.LAUNCH_CONV else act_key(c)
                seen[k] = seen.get(k, 0) + 1

    last = {f: ops.last_launch_config(f)["launches"] for f in (ops.LAUNCH_CONV, ops.LAUNCH_ACT)}
    monkeypatch.setattr(_lib, "check", recording_check)
    wl = bench.make_workload(argparse.Namespace(workload=workload, batch=batch, seconds=seconds), 0)
    model = bench.build_model(wl, DEV)
    with torch.no_grad():
        model(*[t.to(DEV) for t in wl["host_inputs"]])
    torch.cuda.synchronize()
    monkeypatch.setattr(_lib, "check", orig)
    print(f"\n[census] {wl['name']}: " + ", ".join(f"{k} x{n}" for k, n in sorted(seen.items())))
    assert seen, "no conv / activation launch recorded"
    unverified = sorted(set(seen) - VERIFIED)
    assert not unverified, f"{wl['name']} launches variants no case verifies: {unverified}"
