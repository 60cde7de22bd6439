"""The synthesizer front's element-wise, operand-packing, pooling and sampling kernels against float64 at every op and
mode its workloads launch.

test_gpu_front_variants.py covers the front's attention, LayerNorm and conv-epilogue kernels; this file covers the
small fp32 kernels between its convolutions: ``frame_op`` (11 ops), ``pack_blk16_act`` (4 modes), ``wn_res_pack``,
``pack_blk16`` (1-3 addends, leaky_relu, input scale, ragged), ``masked_mean``, ``conv1d_c1_strided``,
``sample_ragged``, ``nearest_gather`` and ``add3_bcast``.  These kernels have no host-side variant choice beyond their
Python arguments, so a call's key is computed from those arguments (``call_key``), both in the cases here and in the
census.

Bounds (u = 2^-24, the fp32 unit roundoff; references in float64 from the kernels' fp32 inputs):
  exact ops          MASK, ADD, FLIP, COUPLE, WN_RES, WN_LAST, ADD_BCAST, ``add3_bcast``, ``nearest_gather``: bit-identical
                     to the fp32 expression in the kernel's order (one correctly rounded fp32 operation per step).
  GATE_ADD           x + (g y) mk: 2 u (|x| + |g y|) -- two roundings, or one if the compiler contracts to an fmaf.
  SAMPLE             m + (e expf(lg)) s: u |m| + 8 u |e exp(lg) s| -- expf <= 2 ulp (<= 4 u relative), two products, the sum.
  GLU_RES            x + y1 sigmoid(y2), sigmoid = 1 / (1 + expf(-y2)): u |x| + 8 u |y1 sigmoid| -- expf 4 u of
                     E = exp(-y2) moves 1 + E by <= 4 u E, the sum 1 + E and the IEEE division add u each, the product u.
  MISH               v tanhf(log1pf(expf(v))) (v for v > 20): 16 u |ref| -- expf 4 u, log1pf <= 1 ulp (2 u), tanhf <= 2
                     ulp (4 u), each relative and carried through slopes <= 1, and the product u.
  packers            half an fp16 ulp of the float64 value plus the fp32 terms of the mode's expression (``_pack_ref``);
                     MASK, ``wn_res_pack`` and ``pack_blk16`` are also bit-identical to fp16(the fp32 expression).
  ``masked_mean``    (ceil(n / 128) + 11) u sum|x| / len: 128 threads each sum ceil(n / 128) frames, 5 shuffle levels, 4
                     warp partials, one division.
  ``conv1d_c1_strided``  (k + 2) u (sum|w x| + |b|): k fmaf steps and the bias add.
Every bound carries 2^-100 (times 1 + |operand| where an expf may underflow) for the fp32 subnormal range.  CPU tests
(f) show each bound fails a plausible defect.  The operand packers, and the LayerNorm, attention and conv kernels that
write blk16 operands, are also checked for the layout's zero padding rows (``padding_violations``).
"""
import argparse
import inspect
import math
import os
import sys

import pytest
import torch
import torch.nn.functional as F

DEV = "cuda:0"
U = 2.0 ** -24
TINY = 2.0 ** -100
BLK_PAD = 32
SENTINEL = 0x7E00                  # an fp16 NaN: what a valid operand row holds before its producer writes it


def _ulp16(a):
    """Spacing of fp16 numbers at |a| (2^-24 in the subnormal range)."""
    return torch.exp2(torch.floor(torch.log2(a.abs().clamp_min(2.0 ** -14))) - 10)


def _cw(C):
    return 64 if C % 64 == 0 else (32 if C % 32 == 0 else 16)


def _prefix_mask(lens, T, device=DEV):
    n = torch.tensor(lens, device=device).clamp(0, T)
    return (torch.arange(T, device=device)[None, :] < n[:, None]).float()


def _mask_lens(B, L, gen):
    """Per-item lengths of a partial mask: a full item, an all-zero item, then random lengths (B = 1: half)."""
    if B == 1:
        return [L // 2]
    extra = torch.randint(0, L + 1, (max(0, B - 2),), generator=gen).tolist()
    return ([L, 0] + extra)[:B]


def _rn(gen, *shape):
    return torch.randn(*shape, generator=gen, device=DEV)


# ----------------------------------------------------------------------------------------------
# call keys: the same function keys the cases below and the census
# ----------------------------------------------------------------------------------------------
FRAME_OPS = {1: "wn_res", 2: "wn_last", 3: "gate_add", 4: "couple", 5: "sample", 6: "mask", 7: "add", 8: "glu_res",
             9: "mish", 10: "flip", 11: "add_bcast"}
PACK_MODES = ("mask", "gate", "gelu", "mish")


def frame_key(op, masked, cform, alias, L):
    """cform: the per-(batch, channel) vector of GATE_ADD / ADD_BCAST, dense (cstride = C) or strided rows; alias: in
    place (out is a), out of place, or WN_LAST's accumulator; th: the launch's thread count (256 from L = 256 on)."""
    return f"frame_op:{FRAME_OPS[op]}:mask{int(masked)}:{cform}:{alias}:th{256 if L >= 256 else 128}"


def pack_act_key(mode, masked, bc, C, prefix):
    return f"pack_blk16_act:{PACK_MODES[mode]}:mask{int(masked)}:bc{int(bc)}:cw{_cw(C)}:{'prefix' if prefix else 'whole'}"


def wn_res_pack_key(masked, C):
    return f"wn_res_pack:mask{int(masked)}:cw{_cw(C)}"


def pack_blk16_key(n, lrelu, scaled, ragged, C):
    return f"pack_blk16:add{n}:lrelu{int(bool(lrelu))}:{'sx' if scaled else 's1'}:vl{int(ragged)}:cw{_cw(C)}"


def masked_mean_key(masked, ragged):
    return f"masked_mean:mask{int(masked)}:vl{int(ragged)}"


def conv_c1_key(k, stride, pad, bias, masked, ragged):
    return f"conv1d_c1_strided:k{k}s{stride}p{pad}:bias{int(bias)}:mask{int(masked)}:vl{int(ragged)}"


def sample_key(seeded, svec, ragged):
    return f"sample_ragged:{'seeded' if seeded else 'eps'}:{'svec' if svec else 's'}:vl{int(ragged)}"


def gather_key(Lin, Lout):
    kind = "same" if Lin == Lout else ("up" if Lout > Lin else ("down-int" if Lin % Lout == 0 else "down-frac"))
    return f"nearest_gather:{kind}"


def add3_key(b, bc, inplace):
    return f"add3_bcast:b{int(b)}:bc{int(bc)}:{'inplace' if inplace else 'oop'}"


def _same(t, u):
    return t is not None and u is not None and t.data_ptr() == u.data_ptr()


def _k_frame(a):
    op, C = a["op"], a["C"]
    alias = "acc" if op == 2 else ("inplace" if _same(a["out"], a["a"]) else "oop")
    cform = "-" if a["c"] is None else ("c=C" if a["cstride"] == C else "c!=C")
    return frame_key(op, a["mask"] is not None, cform, alias, a["L"])


def _k_pack_act(a):
    mode, C, x = a["mode"], a["C"], a["x"]
    need = 2 * C if mode == 1 else C
    return pack_act_key(mode, a["mask"] is not None, a["bcast"] is not None, C, a["c_off"] > 0 or x.shape[1] > need)


def _k_pack(a):
    xs = a["x"] if isinstance(a["x"], (list, tuple)) else [a["x"]]
    return pack_blk16_key(len(xs), a["lrelu"], float(a["scale"]) != 1.0, a["valid_len"] is not None, xs[0].shape[1])


KEYERS = {
    "frame_op": _k_frame,
    "pack_blk16_act": _k_pack_act,
    "wn_res_pack": lambda a: wn_res_pack_key(a["mask"] is not None, a["x"].shape[1]),
    "pack_blk16": _k_pack,
    "masked_mean": lambda a: masked_mean_key(a["mask"] is not None, a["valid_len"] is not None),
    "conv1d_c1_strided": lambda a: conv_c1_key(a["w"].shape[2], a["stride"], a["pad"], a["bias"] is not None,
                                               a["mask"] is not None, a["valid_len"] is not None),
    "sample_ragged": lambda a: sample_key(a["seeds"] is not None, isinstance(a["s"], torch.Tensor),
                                          a["valid_len"] is not None),
    "nearest_gather": lambda a: gather_key(a["x"].shape[-1], a["Lout"]),
    "add3_bcast": lambda a: add3_key(a["b"] is not None, a["bc"] is not None, _same(a["out"], a["a"])),
}


def call_key(fn, name, args, kwargs):
    bound = inspect.signature(fn).bind(*args, **kwargs)
    bound.apply_defaults()
    return KEYERS[name](bound.arguments)


def _call(ops, seen, name, *args, **kwargs):
    """Run ``ops.<name>`` and record the key of the call."""
    fn = getattr(ops, name)
    seen.add(call_key(fn, name, args, kwargs))
    return fn(*args, **kwargs)


# ----------------------------------------------------------------------------------------------
# blk16 padding rows
# ----------------------------------------------------------------------------------------------
def sentinel_buffer(shape, L, device=DEV):
    """A blk16 buffer whose valid rows [BLK_PAD, BLK_PAD + L) hold the sentinel and every other row zero."""
    buf = torch.zeros(shape, dtype=torch.float16, device=device)
    buf.view(torch.int16)[:, :, BLK_PAD:BLK_PAD + L] = SENTINEL
    return buf


def padding_violations(buf, L, vlen=None, bits=True):
    """What a producer did wrong to a ``sentinel_buffer`` (None if nothing): a row outside [BLK_PAD, BLK_PAD + L) is no
    longer zero (the next conv's zero padding), a valid row still holds the sentinel (not written), or -- with ``vlen``
    -- a row of item b at t >= vlen[b] is not zero, as that item's own run leaves it.  ``bits``: those rows must be +0
    (the packers write zero units); else any zero value (an epilogue's act * 0 may give -0)."""
    raw = buf.view(torch.int16)
    if bool((raw[:, :, :BLK_PAD] != 0).any()):
        return "a leading padding row was written"
    if bool((raw[:, :, BLK_PAD + L:] != 0).any()):
        rows = torch.nonzero((raw[:, :, BLK_PAD + L:] != 0).any(-1).any(0).any(0)).flatten()
        return f"a trailing padding row was written (row BLK_PAD + L + {int(rows[0])})"
    valid = raw[:, :, BLK_PAD:BLK_PAD + L]
    if bool((valid == SENTINEL).any()):
        return "a valid row was left unwritten"
    if vlen is not None:
        for b, n in enumerate(vlen):
            n = max(0, min(int(n), L))
            tail = valid[b, :, n:]
            bad = (tail != 0) if bits else ((tail & 0x7FFF) != 0)
            if bool(bad.any()):
                return f"item {b}: a row at t >= valid_len = {n} is not zero"
    return None


# ----------------------------------------------------------------------------------------------
# float64 references and bounds
# ----------------------------------------------------------------------------------------------
def _gate_add_ref(x, y, g, mk):
    p = g * y
    return x + p * mk, 2 * U * (x.abs() + p.abs()) + TINY


def _sample_ref(m, lg, e, s, mk):
    t = e * torch.exp(lg) * s
    return (m + t) * mk, U * (m.abs() + 8 * t.abs()) * mk + TINY


def _glu_ref(x, y1, y2, mk):
    p = y1 * torch.sigmoid(y2)
    return (x + p) * mk, U * (x.abs() + 8 * p.abs()) * mk + TINY * (1 + y1.abs())


def _mish_ref(v, mk):
    ref = v * torch.tanh(F.softplus(v)) * mk             # F.softplus: threshold 20, as the kernel
    return ref, 16 * U * ref.abs() + TINY * (1 + v.abs())


def _pack_ref(mode, x, bc, mk, C):
    """float64 value of a pack_blk16_act mode and its bound: half an fp16 ulp plus the fp32 term (module docstring;
    GATE: tanhf 4 u and its argument's rounding u, sigmoid 7 u and its argument's rounding, which moves sigmoid by
    u |y| (1 - sigmoid) relative; GELU: the polynomial's 7 roundings move tanh by <= 7 u absolute, tanhf 4 u, 1 + tanh u,
    times 0.5 |v|, and the product)."""
    if mode == 1:
        a, g = x[:, :C], x[:, C:2 * C]
        if bc is not None:
            a, g = a + bc[:, :C, None], g + bc[:, C:, None]
        ref = torch.tanh(a) * torch.sigmoid(g)
        A = U * ref.abs() * (16 + g.abs())
    else:
        v = x[:, :C]
        if mode == 0:
            ref, A = v * mk, torch.zeros_like(v)
        elif mode == 2:
            ref = F.gelu(v, approximate="tanh") * mk
            A = (8 * U * v.abs() + 2 * U * ref.abs()) * mk
        else:
            ref, A = _mish_ref(v, mk)
            A = A - TINY * (1 + v.abs())
    return ref, 0.5 * _ulp16(ref) + A + TINY


def _check(got, ref, tol, where):
    err = (got.double() - ref).abs()
    r = float((err / tol).max()) if err.numel() else 0.0
    assert r <= 1.0, (where, r, float(err.max()))
    return r


# ----------------------------------------------------------------------------------------------
# (a) frame_op, all 11 ops
# ----------------------------------------------------------------------------------------------
FRAME_L = (1, 2, 127, 128, 129, 255, 256, 257, 4099)
FRAME_C = (1, 96, 192, 384)
FRAME_B = (1, 3, 17)


def _frame_shapes():
    out = []
    for i, L in enumerate(FRAME_L):
        for j, C in enumerate(FRAME_C):
            B = FRAME_B[(i + j) % 3]
            while B * C * L > 4_000_000 and B > 1:
                B = 3 if B == 17 else 1
            out.append((B, C, L))
    return out


FRAME_SHAPES = _frame_shapes()
EDGE_SHAPE = (3, 96, 257)           # _edge_args needs T >= 32
_IO = (("-", "inplace"), ("-", "oop"))
_VEC = tuple((cf, al) for cf in ("c=C", "c!=C") for al in ("inplace", "oop"))
# op -> (forms (cform, alias) as the call sites and the tests use them, masks)
FRAME_FORMS = {1: (_IO, (0, 1)), 2: ((("-", "acc"),), (0, 1)), 3: (_VEC, (0, 1)), 4: ((("-", "inplace"),), (0, 1)),
               5: ((("-", "oop"),), (0, 1)), 6: (_IO, (0, 1)), 7: (_IO, (0, 1)), 8: (_IO, (0, 1)), 9: (_IO, (0, 1)),
               10: ((("-", "oop"),), (0,)), 11: (_VEC, (0, 1))}
SAMPLE_S = (0.0, 0.333, 1.0)


def _declared_frame(op):
    forms, masks = FRAME_FORMS[op]
    shapes = FRAME_SHAPES + ([EDGE_SHAPE] if op in (5, 8, 9) else [])
    return {frame_key(op, m, cf, al, L) for _, _, L in shapes for cf, al in forms for m in masks}


def _frame_case(ops, seen, op, B, C, L, mask, gen, edge=False):
    """Run every form of ``op`` at one shape and mask; returns the worst error / bound."""
    mk = torch.ones(B, 1, L, device=DEV) if mask is None else mask[:, None, :]
    mk64 = mk.double()
    worst = 0.0
    where = (FRAME_OPS[op], B, C, L, mask is not None, edge)
    forms, _ = FRAME_FORMS[op]
    x = _rn(gen, B, C, L)
    if edge:
        from test_gpu_front import _edge_args
        xe = _edge_args(B, 2 * C, L, torch.Generator().manual_seed(C + L)).to(DEV)
    for cf, al in forms:
        out = torch.full((B, C, L), float("nan"), device=DEV)
        if op == 1:                                         # WN_RES
            rs, o = _rn(gen, B, 2 * C, L), _rn(gen, B, C, L)
            xk, ok = x.clone(), o.clone()
            dst = xk if al == "inplace" else out
            _call(ops, seen, "frame_op", op, xk, rs, None, mask, dst, ok, B, C, L)
            assert torch.equal(dst, (x + rs[:, :C]) * mk), where
            assert torch.equal(ok, o + rs[:, C:]), where
            if al == "oop":
                assert torch.equal(xk, x), where
        elif op == 2:                                       # WN_LAST
            r, o = _rn(gen, B, C, L), _rn(gen, B, C, L)
            ok = o.clone()
            _call(ops, seen, "frame_op", op, None, r, None, mask, None, ok, B, C, L)
            assert torch.equal(ok, (o + r) * mk), where
        elif op in (3, 11):                                 # GATE_ADD, ADD_BCAST
            if cf == "c=C":
                vec, cs = _rn(gen, B, C), C
            else:                                           # a chunk of the batched adaLN output [B, 6C]
                vec, cs = _rn(gen, B, 6 * C)[:, 2 * C:3 * C], 6 * C
            y = _rn(gen, B, C, L)
            xk = x.clone()
            dst = xk if al == "inplace" else out
            _call(ops, seen, "frame_op", op, xk, y if op == 3 else None, vec, mask, dst, None, B, C, L, cstride=cs)
            if op == 11:
                assert torch.equal(dst, (x + vec[:, :, None]) * mk), where
            else:
                ref, tol = _gate_add_ref(x.double(), y.double(), vec.double()[:, :, None], mk64)
                worst = max(worst, _check(dst, ref, tol, where + (cf, al)))
        elif op == 4:                                       # COUPLE
            full, m = _rn(gen, B, 2 * C, L), _rn(gen, B, C, L)
            fk = full.clone()
            _call(ops, seen, "frame_op", op, fk, m, None, mask, fk, None, B, C, L)
            assert torch.equal(fk[:, :C], full[:, :C]) and torch.equal(fk[:, C:], (full[:, C:] - m) * mk), where
        elif op == 5:                                       # SAMPLE
            lg = xe[:, C:] if edge else torch.rand(B, C, L, generator=gen, device=DEV) * 60 - 30
            stats = torch.cat([_rn(gen, B, C, L), lg], 1).contiguous()
            e = _rn(gen, B, C, L)
            for s in SAMPLE_S:
                z = torch.full((B, C, L), float("nan"), device=DEV)
                _call(ops, seen, "frame_op", op, stats, e, None, mask, z, None, B, C, L, s=s)
                ref, tol = _sample_ref(stats[:, :C].double(), stats[:, C:].double(), e.double(), s, mk64)
                # where fp32 overflows (exp(lg) > 3.4e38 or e exp(lg) beyond it) the fp32 expression is what the model
                # computes: inf, or NaN after * 0
                r32 = (stats[:, :C] + (e * torch.exp(stats[:, C:])) * s) * mk
                fin = torch.isfinite(r32)
                assert bool((torch.isnan(z) == torch.isnan(r32)).all()), where + (s,)
                assert bool((z[~fin & ~torch.isnan(z)] == r32[~fin & ~torch.isnan(r32)]).all()), where + (s,)
                worst = max(worst, _check(z[fin], ref[fin], tol[fin], where + (s,)))
        elif op in (6, 7):                                  # MASK, ADD
            y = _rn(gen, B, C, L)
            xk = x.clone()
            dst = xk if al == "inplace" else out
            _call(ops, seen, "frame_op", op, xk, y if op == 7 else None, None, mask, dst, None, B, C, L)
            assert torch.equal(dst, ((x + y) if op == 7 else x) * mk), where
        elif op == 8:                                       # GLU_RES
            y = xe if edge else _rn(gen, B, 2 * C, L) * 4
            xk = x.clone()
            dst = xk if al == "inplace" else out
            _call(ops, seen, "frame_op", op, xk, y, None, mask, dst, None, B, C, L)
            ref, tol = _glu_ref(x.double(), y[:, :C].double(), y[:, C:].double(), mk64)
            worst = max(worst, _check(dst, ref, tol, where + (al,)))
        elif op == 9:                                       # MISH
            v = xe[:, :C].contiguous() if edge else x * 4
            vk = v.clone()
            dst = vk if al == "inplace" else out
            _call(ops, seen, "frame_op", op, vk, None, None, mask, dst, None, B, C, L)
            ref, tol = _mish_ref(v.double(), mk64)
            worst = max(worst, _check(dst, ref, tol, where + (al,)))
        elif op == 10:                                      # FLIP
            _call(ops, seen, "frame_op", op, x, None, None, None, out, None, B, C, L)
            assert torch.equal(out, torch.flip(x, [1])), where
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("op", sorted(FRAME_OPS), ids=[FRAME_OPS[o] for o in sorted(FRAME_OPS)])
def test_frame_op_vs_fp64(hsv, op):
    ops = hsv.ops
    seen, worst = set(), 0.0
    gen = torch.Generator(device=DEV).manual_seed(100 + op)
    hgen = torch.Generator().manual_seed(op)
    masks = FRAME_FORMS[op][1]
    runs = [(s, False) for s in FRAME_SHAPES] + ([(EDGE_SHAPE, True)] if op in (5, 8, 9) else [])
    for (B, C, L), edge in runs:
        for m in masks:
            mask = _prefix_mask(_mask_lens(B, L, hgen), L) if m else None
            worst = max(worst, _frame_case(ops, seen, op, B, C, L, mask, gen, edge))
    torch.cuda.synchronize()
    assert seen == _declared_frame(op), sorted(seen ^ _declared_frame(op))
    print(f"\n[parity] frame_op {FRAME_OPS[op]}: {len(seen)} keys, worst error / bound {worst:.3f}")


# ----------------------------------------------------------------------------------------------
# (b) operand packers
# ----------------------------------------------------------------------------------------------
PACK_C = (16, 32, 48, 64, 192, 384)             # CW = 16 / 32 / 16 / 64 / 64 / 64
PACK_L = (1, 31, 32, 33, 511, 512, 513)         # blk16_rows rounds L up to 512: 1..512 -> 576 rows, 513 -> 1088
# mode -> forms (masked, bcast, prefix)
PACK_ACT_FORMS = {m: tuple((mk, 0, p) for mk in (0, 1) for p in (0, 1)) for m in (0, 2, 3)}
PACK_ACT_FORMS[1] = tuple((0, bc, p) for bc in (0, 1) for p in (0, 1))


def _declared_pack_act(mode):
    return {pack_act_key(mode, m, bc, C, p) for C in PACK_C for m, bc, p in PACK_ACT_FORMS[mode]}


@pytest.mark.gpu
@pytest.mark.parametrize("mode", range(4), ids=PACK_MODES)
def test_pack_blk16_act_vs_fp64(hsv, mode):
    ops = hsv.ops
    seen, worst = set(), 0.0
    gen = torch.Generator(device=DEV).manual_seed(200 + mode)
    B = 3
    for C in PACK_C:
        for L in PACK_L:
            x = _rn(gen, B, 3 * C, L) * 3
            mask = _prefix_mask([L, L // 2, 0], L)
            for m, bc, prefix in PACK_ACT_FORMS[mode]:
                where = (PACK_MODES[mode], C, L, m, bc, prefix)
                need = 2 * C if mode == 1 else C
                c_off = C if (prefix and mode != 1) else 0
                xin = x if prefix else x[:, :need].contiguous()
                bcast = _rn(gen, B, 2 * C) if bc else None
                buf = sentinel_buffer(ops.blk16_shape(B, C, L), L)
                _call(ops, seen, "pack_blk16_act", xin, buf, C, mode, bcast=bcast, mask=mask if m else None,
                      c_off=c_off)
                assert padding_violations(buf, L) is None, (where, padding_violations(buf, L))
                got = ops.unpack_blk16(buf, C, L)
                mk = mask[:, None, :] if m else torch.ones(B, 1, L, device=DEV)
                xs = x[:, c_off:c_off + need]
                if mode == 0:
                    assert torch.equal(got, (xs * mk).half().float()), where
                ref, tol = _pack_ref(mode, xs.double(), None if bcast is None else bcast.double(), mk.double(), C)
                worst = max(worst, _check(got, ref, tol, where))
    assert seen == _declared_pack_act(mode), sorted(seen ^ _declared_pack_act(mode))
    # arguments across softplus's threshold of 20 and deep in tanh / sigmoid saturation
    if mode in (1, 3):
        from test_gpu_front import _edge_args
        C, L = 192, 77
        xe = _edge_args(B, 2 * C, L, torch.Generator().manual_seed(7)).to(DEV)
        buf = sentinel_buffer(ops.blk16_shape(B, C, L), L)
        ops.pack_blk16_act(xe, buf, C, mode)
        assert padding_violations(buf, L) is None
        ref, tol = _pack_ref(mode, xe.double(), None, torch.ones(B, 1, L, device=DEV, dtype=torch.float64), C)
        worst = max(worst, _check(ops.unpack_blk16(buf, C, L), ref, tol, ("edge", PACK_MODES[mode])))
    print(f"\n[parity] pack_blk16_act {PACK_MODES[mode]}: {len(seen)} keys, worst error / bound {worst:.3f}")


WN_BIG = (3, 192, 17000)      # 3 x 24 channel groups x 17000 = 1.22 M units > 148 x 32 CTAs x 256 threads


def _declared_wn_res_pack():
    return {wn_res_pack_key(m, C) for C in PACK_C for m in (0, 1)}


@pytest.mark.gpu
def test_wn_res_pack_vs_fp64(hsv):
    """x = (x + rs[:, :C]) * mask and output += rs[:, C:] bit-identical to fp32, the operand = fp16 of the new x, at every
    CW and across the grid-stride loop."""
    ops = hsv.ops
    seen = set()
    gen = torch.Generator(device=DEV).manual_seed(300)
    shapes = [(3, C, L) for C in PACK_C for L in PACK_L] + [WN_BIG]
    for B, C, L in shapes:
        for m in (0, 1):
            x, rs, o = _rn(gen, B, C, L), _rn(gen, B, 2 * C, L), _rn(gen, B, C, L)
            mask = _prefix_mask([L, L // 2, 0], L) if m else None
            mk = mask[:, None, :] if m else 1.0
            xk, ok = x.clone(), o.clone()
            buf = sentinel_buffer(ops.blk16_shape(B, C, L), L)
            _call(ops, seen, "wn_res_pack", xk, rs, mask, ok, buf)
            where = (B, C, L, m)
            assert padding_violations(buf, L) is None, (where, padding_violations(buf, L))
            x_new = (x + rs[:, :C]) * mk
            assert torch.equal(xk, x_new) and torch.equal(ok, o + rs[:, C:]), where
            assert torch.equal(ops.unpack_blk16(buf, C, L), x_new.half().float()), where
            ref = (x.double() + rs[:, :C].double()) * (mk.double() if m else 1.0)
            _check(ops.unpack_blk16(buf, C, L), ref, 0.5 * _ulp16(ref) + U * ref.abs() + TINY, where)
    assert seen == _declared_wn_res_pack(), sorted(seen ^ _declared_wn_res_pack())
    print(f"\n[parity] wn_res_pack: {len(seen)} keys, bit-identical to fp16 of the fp32 expression")


PACK_SCALES = (1.0, 1.0 / 3.0)


def _pack_lens(L):
    return [L, 0, 1, L // 2, L + 7]             # empty, one frame, half, past the end (clamped)


def _declared_pack_blk16(n):
    return {pack_blk16_key(n, lr, sc != 1.0, rg, C) for C in PACK_C for lr in (0, 1) for sc in PACK_SCALES
            for rg in (0, 1)}


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 3], ids=["one", "two", "three"])
def test_pack_blk16_vs_fp64(hsv, n):
    """((x1 + x2) + x3) * scale [-> leaky_relu 0.1] -> fp16: bit-identical to fp16 of the fp32 expression and within half
    an fp16 ulp + 4 u |scale| sum|x_i| of float64; ragged: rows past each item zero, its frames there never read."""
    ops = hsv.ops
    seen, worst = set(), 0.0
    gen = torch.Generator(device=DEV).manual_seed(400 + n)
    for C in PACK_C:
        for L in PACK_L:
            for ragged in (0, 1):
                lens = _pack_lens(L) if ragged else None
                B = 5 if ragged else 3
                xs = [_rn(gen, B, C, L) for _ in range(n)]
                if ragged:                                   # garbage past each item: must not be read
                    for b, v in enumerate(lens):
                        for t in xs:
                            t[b, :, max(0, v):] = float("nan")
                vl = torch.tensor(lens, dtype=torch.int32, device=DEV) if ragged else None
                valid = _prefix_mask(lens, L)[:, None, :].bool() if ragged else torch.ones(B, 1, L, dtype=torch.bool,
                                                                                             device=DEV)
                for lrelu in (False, True):
                    for sc in PACK_SCALES:
                        where = (n, C, L, ragged, lrelu, sc)
                        buf = sentinel_buffer(ops.blk16_shape(B, C, L), L)
                        _call(ops, seen, "pack_blk16", xs if n > 1 else xs[0], buf, lrelu, scale=sc, valid_len=vl)
                        pv = padding_violations(buf, L, lens)
                        assert pv is None, (where, pv)
                        got = ops.unpack_blk16(buf, C, L)
                        v = xs[0]
                        for t in xs[1:]:
                            v = v + t
                        v = v * sc
                        if lrelu:
                            v = torch.where(v > 0, v, v * 0.1)
                        exp = torch.where(valid, v.half().float(), torch.zeros((), device=DEV))
                        assert torch.equal(got, exp), where
                        s64 = sum(t.double() for t in xs)
                        a64 = sum(t.double().abs() for t in xs)
                        ref = s64 * sc
                        if lrelu:
                            ref = torch.where(ref > 0, ref, 0.1 * ref)
                        ref = torch.where(valid, ref, torch.zeros((), device=DEV, dtype=torch.float64))
                        a64 = torch.where(valid, a64, torch.zeros((), device=DEV, dtype=torch.float64))
                        worst = max(worst, _check(got, ref, 0.5 * _ulp16(ref) + 4 * U * sc * a64 + TINY, where))
    assert seen == _declared_pack_blk16(n), sorted(seen ^ _declared_pack_blk16(n))
    print(f"\n[parity] pack_blk16 {n} addend(s): {len(seen)} keys, worst error / bound {worst:.3f}")


@pytest.mark.gpu
def test_blk16_writers_keep_the_padding_rows(hsv):
    """The LayerNorm / adaLN packers, the tensor-core attention with a blk16 output and the operand-writing conv
    epilogue write exactly the rows [BLK_PAD, BLK_PAD + L) of their operand; with zero_masked / valid_len / a prefix mask
    the rows past each item are zero, as that item's own run leaves them."""
    ops = hsv.ops
    gen = torch.Generator(device=DEV).manual_seed(500)
    B, C = 3, 192
    w = (torch.randn(128, 64, 3, generator=torch.Generator().manual_seed(5)) / 14).to(DEV)
    wp = ops.pack_conv_weight(w, 64)
    bias = _rn(gen, 128)
    for L in PACK_L:
        lens = [L, max(1, L // 2), 0]
        mask = _prefix_mask(lens, L)
        x, y = _rn(gen, B, C, L), _rn(gen, B, C, L)
        mod = _rn(gen, B, 6 * C) * 0.5
        ms = mod.stride(0)
        sh, sc, g = mod[:, :C], mod[:, C:2 * C], mod[:, 2 * C:3 * C]
        for zm in (False, True):
            buf = sentinel_buffer(ops.blk16_shape(B, C, L), L)
            ops.ln_mod_blk16(x, sh, sc, buf, ms, mask, 1e-6, premask=True, zero_masked=zm)
            pv = padding_violations(buf, L, lens if zm else None)
            assert pv is None, ("ln_mod", L, zm, pv)
            buf = sentinel_buffer(ops.blk16_shape(B, C, L), L)
            ops.gate_ln_mod_blk16(x.clone(), y, g, sh, sc, buf, ms, mask, 1e-6, zero_masked=zm)
            pv = padding_violations(buf, L, lens if zm else None)
            assert pv is None, ("gate_ln_mod", L, zm, pv)
        vl = [L, 1, max(1, L // 2)]
        for kw in ({}, {"valid_len": torch.tensor(vl, dtype=torch.int32, device=DEV)}):
            q, k, v = _rn(gen, B, C, L), _rn(gen, B, C, L), _rn(gen, B, C, L)
            buf = sentinel_buffer(ops.blk16_shape(B, C, L), L)
            ops.mha(q, k, v, B, 2, 96, L, L, C * L, C * L, C * L, 96 ** -0.5, False, out_blk=buf, **kw)
            pv = padding_violations(buf, L, vl if kw else None, bits=False)
            assert pv is None, ("mha_blk16", L, bool(kw), pv)
        a = torch.zeros(ops.blk16_shape(B, 64, L), dtype=torch.float16, device=DEV)
        ops.pack_blk16(_rn(gen, B, 64, L), a)
        for mode, mk in ((ops.BLK_NONE, None), (ops.BLK_LRELU, mask)):
            buf = sentinel_buffer(ops.blk16_shape(B, 128, L), L)
            ops.conv1d_umma_blk(a, wp, bias, L, 64, 128, 3, 1, 64, buf, mode, mask=mk)
            pv = padding_violations(buf, L, None if mk is None else lens, bits=False)
            assert pv is None, ("conv1d_umma_blk", L, mode, pv)
    torch.cuda.synchronize()


# ----------------------------------------------------------------------------------------------
# (c) masked_mean and conv1d_c1_strided
# ----------------------------------------------------------------------------------------------
MEAN_L = (1, 127, 128, 129, 10000)


def _mean_tol(a64_sum, n):
    """(ceil(n / 128) + 11) u sum|x| / len for a sum over n frames divided by len."""
    depth = math.ceil(n / 128) + 11
    return depth * U * a64_sum


def _declared_mean():
    return {masked_mean_key(m, r) for m in (0, 1) for r in (0, 1)}


@pytest.mark.gpu
def test_masked_mean_vs_fp64(hsv):
    """Dense: x.sum(2) over ALL frames / mask.sum (StyleEncoder.temporal_avg_pool, frames past the mask hold data); an
    all-zero mask row gives x.sum / 0 = inf as the reference does.  Ragged: item b's mean over its first valid_len[b]
    frames (garbage past them), and NaN for an empty item -- the mean of its own, empty run."""
    ops = hsv.ops
    seen, worst = set(), 0.0
    gen = torch.Generator(device=DEV).manual_seed(600)
    C = 256
    for L in MEAN_L:
        for m in (0, 1):                                    # dense
            B = 3
            x = _rn(gen, B, C, L)
            x[2] = x[2].abs() + 0.5                         # a positive sum under the all-zero mask row: +inf
            lens = [L, max(1, L // 3), 0]
            mask = _prefix_mask(lens, L) if m else None
            got = _call(ops, seen, "masked_mean", x, mask)
            den = mask.double().sum(1, keepdim=True) if m else torch.full((B, 1), float(L), device=DEV,
                                                                           dtype=torch.float64)
            ref = x.double().sum(2) / den
            tol = _mean_tol(x.double().abs().sum(2), L) / den + U * ref.abs() + TINY
            rows = slice(0, 2) if m else slice(0, 3)
            worst = max(worst, _check(got[rows], ref[rows], tol[rows], ("dense", L, m)))
            if m:
                assert bool(torch.isinf(got[2]).all() and (got[2] > 0).all()), ("zero mask row", L)
        for m in (0, 1):                                    # ragged
            lens = [L, 0, 1, L // 2, L + 3]
            B = len(lens)
            x = _rn(gen, B, C, L)
            for b, n in enumerate(lens):
                x[b, :, n:] = float("nan")
            vl = torch.tensor(lens, dtype=torch.int32, device=DEV)
            got = _call(ops, seen, "masked_mean", x, _prefix_mask(lens, L) if m else None, valid_len=vl)
            for b, n in enumerate(lens):
                n = min(n, L)
                if n == 0:
                    assert bool(torch.isnan(got[b]).all()), ("empty item", L)
                    continue
                xb = x[b, :, :n].double()
                ref = xb.sum(1) / n
                tol = _mean_tol(xb.abs().sum(1), n) / n + U * ref.abs() + TINY
                worst = max(worst, _check(got[b], ref, tol, ("ragged", L, m, b, n)))
    assert seen == _declared_mean(), sorted(seen ^ _declared_mean())
    print(f"\n[parity] masked_mean: {len(seen)} keys, worst error / bound {worst:.3f}")


# (B, Cout, Lin, k, stride, pad, bias): PosteriorSFEncoder.pre_filter (9, 4, 4) at Lin % 4 = 0..3, Lin = 1 / 2 (one output
# frame from the pad alone), one shape past the grid cap (4 x 192 x 2000 = 1.5 M outputs) and a second geometry
C1_CASES = [(3, 192, 403, 9, 4, 4, True), (2, 192, 400, 9, 4, 4, True), (2, 192, 401, 9, 4, 4, True),
            (2, 192, 402, 9, 4, 4, True), (1, 16, 1, 9, 4, 4, True), (3, 192, 2, 9, 4, 4, True),
            (4, 192, 8000, 9, 4, 4, True), (2, 64, 37, 5, 2, 0, False)]


def _declared_c1():
    return {conv_c1_key(k, s, p, bias, m, r) for _, _, _, k, s, p, bias in C1_CASES for m in (0, 1) for r in (0, 1)}


@pytest.mark.gpu
def test_conv1d_c1_strided_vs_fp64(hsv):
    ops = hsv.ops
    seen, worst = set(), 0.0
    gen = torch.Generator(device=DEV).manual_seed(700)
    for B0, Cout, Lin, k, s, p, has_bias in C1_CASES:
        w = _rn(gen, Cout, 1, k)
        bias = _rn(gen, Cout) if has_bias else None
        Lout = (Lin + 2 * p - k) // s + 1
        for ragged in (0, 1):
            lens = ([Lout, 0, 1, Lout + 5, max(1, Lout // 2)] if ragged else [Lout, Lout // 2, 0, Lout][:B0])
            B = len(lens)
            x = _rn(gen, B, 1, Lin)
            lin = [min(max(0, min(n, Lout)) * s, Lin) if ragged else Lin for n in lens]
            for b, n in enumerate(lin):                     # past each item's input: never read
                x[b, :, n:] = float("nan")
            t = torch.arange(Lin, device=DEV)
            xz = torch.where(t[None, None, :] < torch.tensor(lin, device=DEV)[:, None, None], x, torch.zeros((), device=DEV))
            for m in (0, 1):
                mask = _prefix_mask(lens, Lout) if m else None
                vl = torch.tensor(lens, dtype=torch.int32, device=DEV) if ragged else None
                got = _call(ops, seen, "conv1d_c1_strided", x, w, bias, s, p, mask=mask, valid_len=vl)
                ref = F.conv1d(xz.double(), w.double(), None if bias is None else bias.double(), stride=s, padding=p)
                absr = F.conv1d(xz.double().abs(), w.double().abs(), None if bias is None else bias.double().abs(),
                                stride=s, padding=p)
                keep = torch.ones(B, 1, Lout, device=DEV, dtype=torch.float64)
                if ragged:
                    keep = keep * _prefix_mask(lens, Lout)[:, None, :].double()
                if m:
                    keep = keep * mask[:, None, :].double()
                ref = ref * keep
                tol = (k + 2) * U * absr + TINY
                where = (B, Cout, Lin, k, s, p, ragged, m)
                worst = max(worst, _check(got, ref, tol, where))
                if ragged:
                    assert bool((got * (1 - _prefix_mask(lens, Lout)[:, None, :]) == 0).all()), where
    assert seen == _declared_c1(), sorted(seen ^ _declared_c1())
    print(f"\n[parity] conv1d_c1_strided: {len(seen)} keys, worst error / bound {worst:.3f}")


# ----------------------------------------------------------------------------------------------
# (d) sample_ragged, nearest_gather, add3_bcast
# ----------------------------------------------------------------------------------------------
SAMPLE_T = (1, 2, 3, 4, 129, 130, 131, 132, 1001)     # T % 4 = 0..3: the last group of 4 frames of a thread


def _declared_sample():
    return {sample_key(sd, sv, rg) for sd in (0, 1) for sv in (0, 1) for rg in (0, 1)}


@pytest.mark.gpu
def test_sample_ragged_vs_fp64(hsv):
    """z = m + n exp(logs) s[b] for t < valid_len[b], else exactly 0 (stats and eps there never read); the seeded path
    equals the eps path fed with ``seeded_normal`` of the same seeds, bit for bit."""
    ops = hsv.ops
    seen, worst = set(), 0.0
    gen = torch.Generator(device=DEV).manual_seed(800)
    for T in SAMPLE_T:
        C = 96 if T > 1000 else 192
        for ragged in (0, 1):
            lens = [T, 0, 1, T // 2, T + 3] if ragged else [T] * 3
            B = len(lens)
            vl = torch.tensor(lens, dtype=torch.int32, device=DEV) if ragged else None
            valid = _prefix_mask(lens, T)[:, None, :].bool()
            stats = torch.cat([_rn(gen, B, C, T), torch.rand(B, C, T, generator=gen, device=DEV) * 60 - 30], 1)
            seeds = torch.randint(0, 2 ** 62, (B,), generator=gen, device=DEV, dtype=torch.int64)
            noise = ops.seeded_normal(seeds, C, T)
            eps = noise.clone()
            if ragged:
                for b, n in enumerate(lens):
                    stats[b, :, n:] = float("nan")
                    eps[b, :, n:] = float("nan")
            svec = torch.tensor([0.0, 0.333, 1.0, 0.5, 2.0][:B], device=DEV)
            for s in (0.333, svec):
                outs = []
                for seeded in (0, 1):
                    kw = {"seeds": seeds} if seeded else {"eps": eps}
                    z = _call(ops, seen, "sample_ragged", stats, s, vl, **kw)
                    outs.append(z)
                    sd = (svec.double()[:, None, None] if isinstance(s, torch.Tensor) else s)
                    m64 = torch.where(valid, stats[:, :C], 0.).double()
                    lg64 = torch.where(valid, stats[:, C:], 0.).double()
                    ref, tol = _sample_ref(m64, lg64, noise.double(), sd, valid.double())
                    where = (T, ragged, seeded, isinstance(s, torch.Tensor))
                    worst = max(worst, _check(z, ref, tol, where))
                    assert bool((z[~valid.expand_as(z)] == 0).all()), where
                assert torch.equal(outs[0], outs[1]), (T, ragged)
    assert seen == _declared_sample(), sorted(seen ^ _declared_sample())
    print(f"\n[parity] sample_ragged: {len(seen)} keys, worst error / bound {worst:.3f}")


# (B, C, Lin, Lout): DBlock's nearest down-sampling by an integer factor (Lout = Lin // factor) at divisible and
# non-divisible Lin, the edges, an up-sampling, and one past the grid cap (128 rows x 12000)
GATHER_CASES = [(2, 64, 400, 100), (2, 64, 403, 100), (3, 32, 4, 1), (1, 16, 1, 1), (2, 128, 7, 3), (2, 8, 5, 12),
                (2, 16, 9, 9), (2, 64, 48000, 12000)]


@pytest.mark.gpu
def test_nearest_gather_values(hsv):
    """Values (not only indices) equal F.interpolate(mode="nearest") on the CPU, bit for bit; at integer factors the source
    index is t * factor exactly."""
    ops = hsv.ops
    seen = set()
    for B, C, Lin, Lout in GATHER_CASES:
        x = torch.randn(B, C, Lin, generator=torch.Generator().manual_seed(Lin + Lout))
        got = _call(ops, seen, "nearest_gather", x.to(DEV), Lout).cpu()
        assert torch.equal(got, F.interpolate(x, size=Lout, mode="nearest")), (B, C, Lin, Lout)
        if Lin % Lout == 0:
            assert torch.equal(got, x[:, :, ::Lin // Lout][:, :, :Lout]), (B, C, Lin, Lout)
    assert seen == {gather_key(c[2], c[3]) for c in GATHER_CASES}
    print(f"\n[parity] nearest_gather: {len(seen)} keys, bit-exact")


ADD3_SHAPES = [(2, 64, 1), (3, 96, 513), (2, 192, 4000)]      # the last past the grid cap (1.5 M elements)


def _declared_add3():
    return {add3_key(b, bc, ip) for b in (0, 1) for bc in (0, 1) for ip in (0, 1)}


@pytest.mark.gpu
def test_add3_bcast_exact(hsv):
    """out = (a + b) + bc[b, c] in that order, b and / or bc absent, in place or not: bit-identical to fp32."""
    ops = hsv.ops
    seen = set()
    gen = torch.Generator(device=DEV).manual_seed(900)
    for B, C, L in ADD3_SHAPES:
        a, b = _rn(gen, B, C, L), _rn(gen, B, C, L)
        bc = _rn(gen, B, C, 1)
        for hb in (0, 1):
            for hbc in (0, 1):
                for ip in (0, 1):
                    ak = a.clone()
                    out = ak if ip else None
                    got = _call(ops, seen, "add3_bcast", ak, b if hb else None, bc if hbc else None, out=out)
                    exp = a
                    if hb:
                        exp = exp + b
                    if hbc:
                        exp = exp + bc
                    assert torch.equal(got, exp), (B, C, L, hb, hbc, ip)
                    if ip:
                        assert got.data_ptr() == ak.data_ptr()
    assert seen == _declared_add3(), sorted(seen ^ _declared_add3())
    print(f"\n[parity] add3_bcast: {len(seen)} keys, bit-exact")


# ----------------------------------------------------------------------------------------------
# (e) census
# ----------------------------------------------------------------------------------------------
FRAME_VERIFIED = set()
FRAME_VERIFIED |= {frame_key(op, m, cf, al, L) for op in (1, 6, 7, 8, 9) for m in (0, 1)
                   for cf, al in (("-", "inplace"), ("-", "oop")) for L in (1, 256)}
FRAME_VERIFIED |= {frame_key(op, m, cf, al, L) for op in (3, 11) for m in (0, 1) for cf in ("c=C", "c!=C")
                   for al in ("inplace", "oop") for L in (1, 256)}
FRAME_VERIFIED |= {frame_key(op, m, "-", al, L) for op, al in ((2, "acc"), (4, "inplace"), (5, "oop")) for m in (0, 1)
                   for L in (1, 256)}
FRAME_VERIFIED |= {frame_key(10, 0, "-", "oop", L) for L in (1, 256)}
FRAME_VERIFIED |= {pack_act_key(mode, m, 0, C, p) for mode in (0, 2, 3) for m in (0, 1) for C in (16, 32, 64)
                   for p in (0, 1)}
FRAME_VERIFIED |= {pack_act_key(1, 0, bc, C, p) for bc in (0, 1) for C in (16, 32, 64) for p in (0, 1)}
FRAME_VERIFIED |= {wn_res_pack_key(m, C) for m in (0, 1) for C in (16, 32, 64)}
FRAME_VERIFIED |= {pack_blk16_key(n, lr, sx, rg, C) for n in (1, 2, 3) for lr in (0, 1) for sx in (0, 1) for rg in (0, 1)
                   for C in (16, 32, 64)}
FRAME_VERIFIED |= {masked_mean_key(m, r) for m in (0, 1) for r in (0, 1)}
FRAME_VERIFIED |= {conv_c1_key(9, 4, 4, 1, m, r) for m in (0, 1) for r in (0, 1)}
FRAME_VERIFIED |= {sample_key(sd, sv, rg) for sd in (0, 1) for sv in (0, 1) for rg in (0, 1)}
FRAME_VERIFIED |= {gather_key(*r) for r in ((400, 100), (403, 100), (5, 12), (9, 9))}
FRAME_VERIFIED |= {add3_key(b, bc, ip) for b in (0, 1) for bc in (0, 1) for ip in (0, 1)}


def _declared_frame_keys():
    """The keys the cases of (a)-(d) run (each GPU test asserts it ran exactly its declared keys)."""
    keys = set()
    for op in FRAME_OPS:
        keys |= _declared_frame(op)
    for mode in range(4):
        keys |= _declared_pack_act(mode)
    keys |= _declared_wn_res_pack()
    for n in (1, 2, 3):
        keys |= _declared_pack_blk16(n)
    keys |= _declared_mean() | _declared_c1() | _declared_sample() | _declared_add3()
    keys |= {gather_key(c[2], c[3]) for c in GATHER_CASES}
    return keys


def test_frame_verified_set_is_covered_by_the_cases():
    missing = FRAME_VERIFIED - _declared_frame_keys()
    assert not missing, sorted(missing)


def test_frame_cases_reach_every_edge():
    """Both frame_op thread counts with every C and B, CW = 16 / 32 / 64 in the packers, the 512-row rounding of the
    operand, and the grid-stride loops (> 148 x 32 CTAs x 256 threads) of wn_res_pack, conv1d_c1_strided,
    nearest_gather and add3_bcast."""
    cap = 148 * 32 * 256
    assert {C for _, C, _ in FRAME_SHAPES} == set(FRAME_C) and {B for B, _, _ in FRAME_SHAPES} == set(FRAME_B)
    for th in (128, 256):
        assert {C for _, C, L in FRAME_SHAPES if (L >= 256) == (th == 256)} == set(FRAME_C)
    assert {_cw(C) for C in PACK_C} == {16, 32, 64}
    assert {L <= 512 for L in PACK_L} == {True, False}
    assert WN_BIG[0] * WN_BIG[1] // 8 * WN_BIG[2] > cap
    assert any(B * C * ((Lin + 2 * p - k) // s + 1) > cap for B, C, Lin, k, s, p, _ in C1_CASES)
    assert any(B * C * Lout > cap for B, C, _, Lout in GATHER_CASES)
    assert any(B * C * L > cap for B, C, L in ADD3_SHAPES)
    assert {T % 4 for T in SAMPLE_T} == {0, 1, 2, 3}


CALLS = tuple(KEYERS)


def _record_frame(hsv, monkeypatch, run):
    """Keys of every call of the wrapped ``ops`` functions during ``run``."""
    ops = hsv.ops
    seen = {}

    def wrap(name, fn):
        def rec(*args, **kwargs):
            k = call_key(fn, name, args, kwargs)
            seen[k] = seen.get(k, 0) + 1
            return fn(*args, **kwargs)
        return rec

    origs = {n: getattr(ops, n) for n in CALLS}
    for n, fn in origs.items():
        monkeypatch.setattr(ops, n, wrap(n, fn))
    try:
        with torch.no_grad():
            run()
        torch.cuda.synchronize()
    finally:
        for n, fn in origs.items():
            monkeypatch.setattr(ops, n, fn)
    return seen


def _assert_census(name, seen, calls=True):
    """``calls=False``: a model that launches none of these kernels (SpeechSR48: its convs take the fused activation
    path) -- any call it starts making must still be a verified one."""
    print(f"\n[census] {name} frame kernels: " + (", ".join(f"{k} x{n}" for k, n in sorted(seen.items())) or "none"))
    assert seen or not calls, f"{name}: no frame-kernel call recorded"
    unverified = sorted(set(seen) - FRAME_VERIFIED)
    assert not unverified, f"{name} calls frame-kernel forms no case verifies: {unverified}"


CENSUS = [("synth", 1, 10.0), ("tts", 1, 10.0), ("vocoder", 16, 10.0), ("speechsr48", 16, 10.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("workload,batch,seconds", CENSUS, ids=[f"{w}-B{b}" for w, b, _ in CENSUS])
def test_census_workload_frame_verified(hsv, monkeypatch, workload, batch, seconds):
    """One eager forward of a benchmark workload (bench.py's model and inputs)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    import bench

    wl = bench.make_workload(argparse.Namespace(workload=workload, batch=batch, seconds=seconds), 0)
    model = bench.build_model(wl, DEV)
    seen = _record_frame(hsv, monkeypatch, lambda: model(*[t.to(DEV) for t in wl["host_inputs"]]))
    _assert_census(wl["name"], seen, calls=workload != "speechsr48")


def _lens(lens):
    return torch.tensor(lens, dtype=torch.int32, device=DEV)


@pytest.mark.gpu
def test_census_ragged_batches_frame_verified(hsv, monkeypatch):
    """Ragged vocoder, SpeechSR48 and text-to-vec tail batches."""
    from conftest import golden_sd
    from oracle import synth
    voc = hsv.Vocoder()
    voc.load_state_dict(synth.vocoder_sd(1234), strict=True)
    voc.to(DEV).eval()
    lens = [500, 1, 2, 37, 499, 250]
    z, g = synth.vocoder_inputs(len(lens), max(lens), seed=21)
    _assert_census(f"ragged vocoder B={len(lens)}",
                   _record_frame(hsv, monkeypatch, lambda: voc(z.to(DEV), g.to(DEV), lengths=_lens(lens))))
    sr = hsv.SpeechSR48(100, 40, **hsv.SR_CFG)
    sr.load_state_dict(golden_sd("speechsr48_state.npz"), strict=True)
    sr.to(DEV).eval()
    lens = [48000, 1, 7, 16001, 3333]
    x = torch.randn(len(lens), 1, max(lens), generator=torch.Generator().manual_seed(48)) * 0.3
    _assert_census(f"ragged SpeechSR48 B={len(lens)}",
                   _record_frame(hsv, monkeypatch, lambda: sr(x.to(DEV), lengths=_lens(lens))), calls=False)
    tail = hsv.TTVTail()
    tail.load_state_dict(synth.ttv_tail_sd(3456), strict=True)
    tail.to(DEV).eval()
    lens = [333, 300, 129, 1, 2]
    z, _, g = synth.ttv_tail_inputs(len(lens), max(lens), seed=22)
    _assert_census(f"ragged text-to-vec tail B={len(lens)}",
                   _record_frame(hsv, monkeypatch, lambda: tail(z.to(DEV), None, g.to(DEV), lengths=_lens(lens))))


@pytest.mark.gpu
def test_census_per_item_synthesizer_frame_verified(hsv, monkeypatch):
    """A per-item synthesizer batch of 16 mixed source and prompt lengths, padded as runtime.ragged_prompt_batches pads
    them, with per-item seeds and noise scales."""
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
        for kw in ({}, {"seed": torch.arange(B, dtype=torch.int64, device=DEV) + 7}):
            s = _record_frame(hsv, monkeypatch, lambda: model.voice_conversion_noise_control(
                src.to(DEV), vl, mel.to(DEV), tl, f0.to(DEV), 0.333, False, 0.3, per_item=True, **kw))
            for k, c in s.items():
                seen[k] = seen.get(k, 0) + c
    _assert_census(f"per-item synthesizer B={n} ({len(batches)} batches)", seen)


# ----------------------------------------------------------------------------------------------
# (f) CPU negative controls: each bound fails a plausible defect
# ----------------------------------------------------------------------------------------------
def _ratio(got, ref, tol):
    r = (got.double() - ref).abs() / tol
    return float(torch.nan_to_num(r, nan=float("inf")).max())


def _sigmoid32(v):
    return 1.0 / (1.0 + torch.exp(-v))


def test_frame_bounds_fail_an_fp16_intermediate():
    """The fp32 expressions of GATE_ADD / SAMPLE / GLU_RES, emulated in fp32 on the CPU, pass their bounds; the same with
    the product rounded to fp16 before the sum and the mask fails them."""
    gen = torch.Generator().manual_seed(11)
    B, C, L = 2, 96, 300
    x, y, y2 = (torch.randn(B, C, L, generator=gen) for _ in range(3))
    g = torch.randn(B, C, 1, generator=gen)
    lg = torch.rand(B, C, L, generator=gen) * 60 - 30
    mk = _prefix_mask([L, L // 2], L, "cpu")[:, None, :]
    h = lambda t: t.half().float()
    cases = {
        "gate_add": (lambda r: x + r(g * y) * mk, _gate_add_ref(x.double(), y.double(), g.double(), mk.double())),
        "sample": (lambda r: (x + r(y * torch.exp(lg)) * 0.333) * mk,
                   _sample_ref(x.double(), lg.double(), y.double(), 0.333, mk.double())),
        "glu_res": (lambda r: (x + r(y * _sigmoid32(y2))) * mk, _glu_ref(x.double(), y.double(), y2.double(), mk.double())),
    }
    for name, (emu, (ref, tol)) in cases.items():
        ok, bad = _ratio(emu(lambda t: t), ref, tol), _ratio(emu(h), ref, tol)
        print(f"\n[bound] {name}: error / bound  fp32 {ok:.3f}  fp16 intermediate {bad:.1f}")
        assert ok <= 1.0 < bad, (name, ok, bad)


def _mish32(v, cmp):
    sp = torch.where(cmp(v), v, torch.log1p(torch.exp(v)))
    return v * torch.tanh(sp)


def test_mish_bound_fails_a_softplus_threshold_on_the_wrong_side():
    """The kernel's mish (softplus = v for v > 20) emulated in fp32 passes the MISH bound; taking softplus = v on the
    wrong side of the threshold (v < 20) fails it.  ``v >= 20`` instead of ``v > 20`` is an equivalent mutant in fp32:
    at v = 20, log1p(exp(20)) = 20 + 2e-9 rounds to 20, and tanhf of anything above ~9 is 1 -- no output can show it."""
    from test_gpu_front import _edge_args
    v = _edge_args(2, 96, 300, torch.Generator().manual_seed(12))
    ref, tol = _mish_ref(v.double(), torch.ones(1, 1, 1, dtype=torch.float64))
    ok = _ratio(_mish32(v, lambda t: t > 20), ref, tol)
    bad = _ratio(_mish32(v, lambda t: t < 20), ref, tol)
    print(f"\n[bound] mish: error / bound  fp32 {ok:.3f}  threshold on the wrong side {bad:.1f}")
    assert ok <= 1.0 < bad, (ok, bad)
    assert torch.equal(_mish32(v, lambda t: t >= 20), _mish32(v, lambda t: t > 20))


def test_pack_bound_fails_an_fp16_input():
    """The GELU / MISH packer's bound (half an fp16 ulp + the fp32 term) passes the kernel's expression in fp32 and fails
    the same with its input rounded to fp16 first (two fp16 roundings)."""
    gen = torch.Generator().manual_seed(13)
    B, C, L = 2, 64, 500
    x = torch.randn(B, C, L, generator=gen) * 3
    k = 0.7978845608028654
    emus = {2: lambda v: 0.5 * v * (1.0 + torch.tanh(k * (v + 0.044715 * v * v * v))),
            3: lambda v: _mish32(v, lambda t: t > 20)}
    one = torch.ones(B, 1, L, dtype=torch.float64)
    for mode, emu in emus.items():
        ref, tol = _pack_ref(mode, x.double(), None, one, C)
        ok = _ratio(emu(x).half().float(), ref, tol)
        bad = _ratio(emu(x.half().float()).half().float(), ref, tol)
        print(f"\n[bound] pack {PACK_MODES[mode]}: error / bound  fp32 {ok:.3f}  fp16 input {bad:.2f}")
        assert ok <= 1.0 < bad, (mode, ok, bad)


@pytest.mark.parametrize("L", PACK_L)
def test_padding_check_catches_a_one_row_overrun(L):
    """``padding_violations`` passes a packer that writes exactly the valid rows (and zeros past each item of a ragged
    pack) and catches one that writes one row too many or too few, one row early, or leaves an item's tail."""
    shape = (3, 2, 64 + ((L + 511) // 512) * 512, 32)

    def packed(first, last, tail_from=None):
        buf = sentinel_buffer(shape, L, "cpu")
        buf.view(torch.int16)[:, :, BLK_PAD + first:BLK_PAD + last] = 0x3C00      # 1.0
        if tail_from is not None:
            for b, n in enumerate(tail_from):
                buf.view(torch.int16)[b, :, BLK_PAD + n:BLK_PAD + L] = 0
        return buf

    lens = [L, 0, L // 2]
    assert padding_violations(packed(0, L), L) is None
    assert padding_violations(packed(0, L, lens), L, lens) is None
    assert "trailing padding row" in padding_violations(packed(0, L + 1), L)          # t <= L
    assert "leading padding row" in padding_violations(packed(-1, L), L)
    assert "left unwritten" in padding_violations(packed(0, L - 1), L)
    assert "not zero" in padding_violations(packed(0, L), L, lens)                   # ragged tail written


def test_masked_mean_bound_fails_summing_only_the_masked_frames():
    """The reference divides the sum over ALL frames by the mask sum; a kernel that summed only the frames under the mask
    (dividing by the same count) fails the bound as soon as frames past the mask hold data."""
    gen = torch.Generator().manual_seed(14)
    B, C, L = 2, 256, 1000
    x = torch.randn(B, C, L, generator=gen, dtype=torch.float64)
    lens = [L, 600]
    den = torch.tensor(lens, dtype=torch.float64)[:, None]
    ref = x.sum(2) / den
    tol = _mean_tol(x.abs().sum(2), L) / den + U * ref.abs() + TINY
    ok = _ratio(x.float().sum(2).double() / den, ref, tol)
    bad = _ratio(torch.stack([x[b, :, :n].sum(1) for b, n in enumerate(lens)]) / den, ref, tol)
    print(f"\n[bound] masked_mean: error / bound  fp32 sum {ok:.3f}  masked frames only {bad:.1f}")
    assert ok <= 1.0 < bad, (ok, bad)
