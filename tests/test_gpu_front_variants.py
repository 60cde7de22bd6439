"""The synthesizer front's kernels against a float64 reference at every variant its workloads launch.

test_gpu_variants.py does this for the vocoder's conv and activation kernels; the front runs on three more: the
tensor-core attention (csrc/mha_mma.cu), the LayerNorm / adaLN operand packers (csrc/frame_ops.cu) and the
operand-writing epilogue of the tcgen05 conv (csrc/conv_umma.cu).  Every case reads back, through
``ops.last_launch_config``, the variant it ran, and compares with float64 computed on the device from the kernel's fp32
inputs; where the kernel rounds an operand to fp16 by design, the reference rounds it too.

(a) attention: head dims, output modes, the three masking forms and both staging paths of K / V and Q (16-byte or
    4-byte copies), at the key-split boundaries of the cluster and in four logit regimes.  Bound: 1e-3 x max|V| of the
    (batch, head) slice, over the whole output; rows past ``valid_len`` exactly 0.  A CPU test shows the bound tells
    the hi / lo split logits of the kernel from plain fp16 logits.
(b) LayerNorm / adaLN packers: all 16 instantiations, within one fp16 ulp plus the fp32 term derived in
    ``_ln_ref``; a CPU test shows a one-pass variance fails that bound.
(c) the operand-writing epilogue: every mode at every n_tile, within one fp16 ulp plus the conv's fp32 term.
(d) census: the attention variant of every launch of the synth and tts workloads and of a per-item synthesizer batch
    must be one (a) verifies.
"""
import argparse
import os
import sys

import pytest
import torch
import torch.nn.functional as F

DEV = "cuda:0"
U32 = 2.0 ** -24            # unit roundoff of fp32


def _ulp16(a):
    """Spacing of fp16 numbers at |a| (2^-24 in the subnormal range)."""
    return torch.exp2(torch.floor(torch.log2(a.abs().clamp_min(2.0 ** -14))) - 10)


def _ulp32(a):
    return torch.exp2(torch.floor(torch.log2(a.abs().clamp_min(2.0 ** -126))) - 23)


def _prefix_mask(lens, T, device):
    return (torch.arange(T, device=device)[None, :] < torch.tensor(lens, device=device)[:, None]).float()


# ----------------------------------------------------------------------------------------------
# (a) attention
# ----------------------------------------------------------------------------------------------
# (D, output, masking form, prescale): timm (DiT) scales after the product, the StyleEncoder before it with
# masked_fill(-1e4) over ``lens``; per-item batches give both their ``valid_len``
ATTN_CASES = [(D, out, form, pre) for D in (96, 128) for out in ("f32", "blk16")
              for form, pre in (("none", False), ("lens", True), ("vlen", False), ("vlen", True))]
ATTN_CASES.append((64, "f32", "none", False))   # the C-ABI takes D = 64 too
# 1..17: one key tile (CTA 1 of the cluster idle); 64 / 65: 4 / 5 tiles (whether CTA 1 gets one); 127..129: every
# warp stream holds one tile or one holds two; 150 / 500: the workloads; 1500: a 30 s utterance
ATTN_T = (1, 15, 16, 17, 64, 65, 127, 128, 129, 150, 500, 1500)
REGIMES = ("randn", "x16", "ramp", "equal")
# (q offset, k / v offset) in floats: a view one float into its buffer takes the 4-byte staging path
STAGING_T = (64, 500)
STAGING = ((1, 0), (0, 1))
HEADS = 2
ATTN_GARBAGE = 1.0e3


def mha_key(c):
    """Variant key of an attention launch from its ``last_launch_config`` record."""
    if c["kernel"]:
        return "mha:fp32-cuda-core"
    form = "vlen" if c["has_valid_len"] else ("lens" if c["has_lens"] else "none")
    return (f"mha:d{c['D']}:{'blk16' if c['out_mode'] else 'f32'}:{form}:{'pre' if c['prescale'] else 'post'}"
            f":kv{c['kv16']}:q{c['q16']}")


def _mha_key_expected(D, out, form, pre, kv16, q16):
    return f"mha:d{D}:{out}:{form}:{'pre' if pre else 'post'}:kv{int(kv16)}:q{int(q16)}"


def _attn_runs(D):
    """(T, regime, q offset, kv offset) of one case: every T and regime aligned, the misaligned views at STAGING_T."""
    runs = [(T, r, 0, 0) for T in ATTN_T for r in REGIMES]
    runs += [(T, r, qo, ko) for T in STAGING_T for r in ("randn", "x16") for qo, ko in STAGING]
    return runs


def _staging(T, qo, ko):
    return T % 4 == 0 and ko == 0, T % 4 == 0 and qo == 0


def _attn_batch(T):
    return 16 if T <= 150 else (4 if T <= 500 else 2)


def _attn_lens(T, B, gen):
    extra = torch.randint(1, T + 1, (max(0, B - 2),), generator=gen).tolist()
    return ([T, 1] + extra)[:B]


def _attn_inputs(B, D, T, regime, scale, gen):
    """q, k, v [B, HEADS*D, T] fp32 (CPU) of a logit regime."""
    C = HEADS * D
    q, k, v = (torch.randn(B, C, T, generator=gen) for _ in range(3))
    if regime == "x16":                       # logits x16: a peaked softmax
        q *= 16
    elif regime == "ramp":                    # logit t / 16 added at key t: the running max rises in every key tile
        for h in range(HEADS):
            q[:, h * D] = 2.0
            k[:, h * D] = torch.arange(T, dtype=torch.float32) / (16 * 2.0 * scale)
    elif regime == "equal":                   # every key the same: all logits of a row equal
        k = k[:, :, :1].expand(B, C, T).contiguous()
    return q, k, v


def _attn_ref(q, k, v, B, D, T, scale, form, lens):
    """float64 attention on the device; V rounded to fp16 as the kernel's P V operand.  [B, HEADS, D, T]."""
    q64, k64 = (t.double().view(B, HEADS, D, T) for t in (q, k))
    v64 = v.half().double().view(B, HEADS, D, T)
    s = torch.einsum("bhdi,bhdj->bhij", q64, k64) * scale
    if form == "lens":
        m = _prefix_mask(lens, T, q.device).double()
        s = s.masked_fill((m[:, None, :, None] * m[:, None, None, :]) == 0, -1e4)
    elif form == "vlen":
        m = _prefix_mask(lens, T, q.device)
        s = s.masked_fill(m[:, None, None, :] == 0, float("-inf"))
    out = torch.einsum("bhij,bhdj->bhdi", s.softmax(-1), v64)
    if form == "vlen":
        out = out * m[:, None, None, :].double()
    return out


def _attn_bound(v, B, D, T, form, lens):
    """1e-3 x max|V| of each (b, h) slice over the keys the item attends to: [B, HEADS, 1, 1]."""
    va = v.half().double().abs().view(B, HEADS, D, T)
    if form == "vlen":
        va = va * _prefix_mask(lens, T, v.device).double()[:, None, None, :]
    return 1e-3 * va.amax(dim=(2, 3), keepdim=True)


def _view(x, off):
    """x [B, C, T] copied into a flat buffer starting ``off`` floats in (off = 1: not 16-byte aligned)."""
    buf = torch.zeros(x.numel() + 4, device=DEV)
    buf[off:off + x.numel()] = x.reshape(-1).to(DEV)
    return buf[off:off + x.numel()]


@pytest.mark.gpu
@pytest.mark.parametrize("D,out,form,pre", ATTN_CASES, ids=[f"d{c[0]}-{c[1]}-{c[2]}-{'pre' if c[3] else 'post'}"
                                                            for c in ATTN_CASES])
def test_mha_vs_fp64(hsv, D, out, form, pre):
    ops = hsv.ops
    ops.set_mha_variant(0)
    C, scale = HEADS * D, D ** -0.5
    seen, worst = set(), 0.0
    for i, (T, regime, qo, ko) in enumerate(_attn_runs(D)):
        gen = torch.Generator().manual_seed(1000 * D + 7 * T + i)
        B = _attn_batch(T)
        q, k, v = _attn_inputs(B, D, T, regime, scale, gen)
        lens = _attn_lens(T, B, gen) if form != "none" else None
        if form == "vlen":                    # frames past an item are never read: garbage there would show
            for b, n in enumerate(lens):
                for t in (q, k, v):
                    t[b, :, n:] = ATTN_GARBAGE * (torch.rand(C, T - n, generator=gen) - 0.5)
        qd, kd, vd = _view(q, qo), _view(k, ko), _view(v, ko)
        kw = {}
        if form == "lens":
            kw["lens"] = torch.tensor(lens, dtype=torch.int32, device=DEV)
        elif form == "vlen":
            kw["valid_len"] = torch.tensor(lens, dtype=torch.int32, device=DEV)
        if out == "blk16":
            buf = torch.zeros(ops.blk16_shape(B, C, T), dtype=torch.float16, device=DEV)
            ops.mha(qd, kd, vd, B, HEADS, D, T, T, C * T, C * T, C * T, scale, pre, out_blk=buf, **kw)
            rec = ops.last_launch_config(ops.LAUNCH_MHA)
            got = ops.unpack_blk16(buf, C, T)
        else:
            got = ops.mha(qd, kd, vd, B, HEADS, D, T, T, C * T, C * T, C * T, scale, pre, **kw)
            rec = ops.last_launch_config(ops.LAUNCH_MHA)
        key = mha_key(rec)
        assert key == _mha_key_expected(D, out, form, pre, *_staging(T, qo, ko)), (T, regime, qo, ko, key)
        assert (rec["key_tiles"], rec["grid_x"], rec["grid_y"], rec["grid_z"]) == (-(-T // 16), -(-T // 16), 2 * HEADS, B)
        seen.add(key)
        qc, kc, vc = (t.to(DEV) for t in (q, k, v))
        ref = _attn_ref(qc, kc, vc, B, D, T, scale, form, lens)
        got = got.double().view(B, HEADS, D, T)
        tol = _attn_bound(vc, B, D, T, form, lens).expand_as(ref)
        if out == "blk16":
            tol = tol + 0.5 * _ulp16(ref)
        err = (got - ref).abs()
        worst = max(worst, float((err / tol).max()))
        bad = err > tol
        assert not bool(bad.any()), (T, regime, qo, ko, float((err / tol).max()),
                                     [int(i) for i in torch.nonzero(bad)[0]])
        if form == "vlen":
            for b, n in enumerate(lens):
                assert bool((got[b, :, :, n:] == 0).all()), (T, regime, b, n)
    assert seen == {_mha_key_expected(D, out, form, pre, kv, qq) for kv in (0, 1) for qq in (0, 1)}, seen
    print(f"\n[parity] mha d{D} {out} {form} {'pre' if pre else 'post'}: worst error / bound {worst:.3f}")


def _emulate_mha(q, k, v, scale, hilo):
    """The tensor-core kernel's rounding in float64 (CPU): logits from fp16 hi / lo halves of q and k (``hilo``) or from
    plain fp16 q and k; P and V rounded to fp16 before P V, the sum divided by the unrounded row sum.  [.., D, T]."""
    h = lambda t: t.half().double()
    q, k = q.float(), k.float()
    qh, kh = h(q), h(k)
    s = torch.einsum("...di,...dj->...ij", qh, kh)
    if hilo:
        ql, kl = h(q - q.half().float()), h(k - k.half().float())
        s = s + torch.einsum("...di,...dj->...ij", qh, kl) + torch.einsum("...di,...dj->...ij", ql, kh)
    s = s * scale
    p = torch.exp(s - s.amax(-1, keepdim=True))
    return torch.einsum("...ij,...dj->...di", h(p), h(v)) / p.sum(-1)[..., None, :]


@pytest.mark.parametrize("T", [150, 500])
def test_attention_bound_tells_hilo_logits_from_plain_fp16(T):
    """At the x16 regime the bound of (a) passes the hi / lo split logits of the kernel's design and fails plain fp16
    logits; if it passed both, it could not see the kernel lose the split."""
    D, B = 96, 2
    scale = D ** -0.5
    q, k, v = _attn_inputs(B, D, T, "x16", scale, torch.Generator().manual_seed(T))
    shape = (B, HEADS, D, T)
    ref = _attn_ref(q, k, v, B, D, T, scale, "none", None)
    bound = _attn_bound(v, B, D, T, "none", None)
    ratio = {}
    for hilo in (True, False):
        got = _emulate_mha(q.view(shape), k.view(shape), v.view(shape), scale, hilo)
        ratio[hilo] = float(((got - ref).abs() / bound).max())
    print(f"\n[bound] attention T={T}: error / bound  hi/lo {ratio[True]:.3f}  plain fp16 {ratio[False]:.3f}")
    assert ratio[True] < 1.0 < ratio[False], ratio


# ----------------------------------------------------------------------------------------------
# (b) LayerNorm / adaLN operand packers
# ----------------------------------------------------------------------------------------------
LN_C = (64, 128, 192, 256)
LN_T = (1, 31, 32, 33, 500, 1500)       # CTAs of 32 steps: a ragged last CTA at 1, 31, 33, 500, 1500
LN_INPUTS = (("mean300-std0.5", 300.0, 0.5), ("mean1-std3", 1.0, 3.0), ("randn", 0.0, 1.0))
LN_EPS = 1e-6


def _ln_ref(x, y, gate, shift, scale, mask, inmask, premask, zero_masked):
    """float64 LayerNorm (no affine) -> modulate, and the bound of the fp16 operand.  Returns (x_new, out, tol).

    The kernel's fp32 path: mean = fl(sum) / C with each thread summing its CPT = C / 8 channels in order, then the 8
    partial sums in order -- at most CPT + 8 rounded steps, so |mean error| <= (CPT + 8) u M (u = 2^-24, M = the row's
    max |value|; a fused gate update adds u M to each value).  The mean error moves every centred value d by the same
    amount: times rstd and |1 + scale| in the output.  The centred sum of squares, rsqrtf, the product with rstd and
    the modulation add a few u relative to |nrm (1 + scale)| and |shift|.  So the fp32 value is within
    A = (CPT + 16) u (M rstd |1 + scale| + |nrm (1 + scale)| + |shift|) of the float64 one, and rounding it to fp16
    moves it by at most half an fp16 ulp: bound = ulp16(ref) + A.  A one-pass variance E[x^2] - E[x]^2 loses
    (E[x^2] / var) u relative, far outside A when |mean| >> std."""
    B, C, T = x.shape
    mk = mask.double()[:, None, :]
    x64 = x.double()
    upd = torch.zeros_like(x64)
    if y is not None:
        upd = gate.double()[:, :, None] * y.double() * mk
        x64 = x64 + upd
    v = x64 * mk if inmask else x64
    mean = v.mean(1, keepdim=True)
    d = v - mean
    rstd = 1.0 / torch.sqrt((d * d).mean(1, keepdim=True) + LN_EPS)
    nrm = d * rstd
    if premask:
        nrm = nrm * mk
    s1 = 1.0 + scale.double()[:, :, None]
    sh = shift.double()[:, :, None]
    out = nrm * s1 + sh
    if zero_masked:
        out = out * mk
    M = torch.maximum(v.abs(), upd.abs()).amax(1, keepdim=True)
    A = (C // 8 + 16) * U32 * (M * rstd * s1.abs() + (nrm * s1).abs() + sh.abs())
    return x64, out, _ulp16(out) + A


@pytest.mark.gpu
@pytest.mark.parametrize("zero_masked", [False, True], ids=["plain", "zero-masked"])
@pytest.mark.parametrize("fused", [False, True], ids=["ln_mod", "gate_ln_mod"])
@pytest.mark.parametrize("C", LN_C)
def test_ln_mod_vs_fp64(hsv, C, fused, zero_masked):
    ops = hsv.ops
    B, worst = 3, 0.0
    for T in LN_T:
        mask = _prefix_mask([T, max(1, T // 2), 0], T, DEV)                 # a partial and an all-zero item
        for name, mu, sd in LN_INPUTS:
            gen = torch.Generator().manual_seed(C + 31 * T + int(mu))
            x = (torch.randn(B, C, T, generator=gen) * sd + mu).to(DEV)
            y = torch.randn(B, C, T, generator=gen).to(DEV)
            mod = (torch.randn(B, 3, 6 * C, generator=gen) * 0.5).to(DEV)[:, 1]   # strided rows of the adaLN output
            ms = mod.stride(0)
            shift, scale, gate = mod[:, :C], mod[:, C:2 * C], mod[:, 2 * C:3 * C]
            for premask in (False, True):
                for inmask in ((False,) if fused else (False, True)):
                    buf = torch.zeros(ops.blk16_shape(B, C, T), dtype=torch.float16, device=DEV)
                    xk = x.clone()
                    if fused:
                        ops.gate_ln_mod_blk16(xk, y, gate, shift, scale, buf, ms, mask, LN_EPS, premask=premask,
                                              zero_masked=zero_masked)
                    else:
                        ops.ln_mod_blk16(xk, shift, scale, buf, ms, mask, LN_EPS, inmask=inmask, premask=premask,
                                         zero_masked=zero_masked)
                    x_new, ref, tol = _ln_ref(x, y if fused else None, gate, shift, scale, mask, inmask, premask,
                                              zero_masked)
                    got = ops.unpack_blk16(buf, C, T).double()
                    where = (T, name, premask, inmask)
                    err = (got - ref).abs()
                    worst = max(worst, float((err / tol).max()))
                    assert bool((err <= tol).all()), (where, float((err / tol).max()))
                    if zero_masked:
                        assert bool((got * (1 - mask[:, None, :].double()) == 0).all()), where
                    if fused:            # the fused x += gate * y * mask: two fp32 roundings, each half an ulp
                        upd = (gate.double()[:, :, None] * y.double() * mask[:, None, :].double()).abs()
                        xe = (xk.double() - x_new).abs()
                        assert bool((xe <= _ulp32(torch.maximum(x_new.abs(), upd))).all()), (where, float(xe.max()))
                    else:
                        assert torch.equal(xk, x), where
                    raw = buf.view(-1, buf.shape[-2], buf.shape[-1])
                    assert float(raw[:, :ops.BLK_PAD].abs().max()) == 0.0
                    assert float(raw[:, ops.BLK_PAD + T:].abs().max()) == 0.0
    print(f"\n[parity] {'gate_ln_mod' if fused else 'ln_mod'} C={C} zero_masked={zero_masked}: worst error / bound "
          f"{worst:.3f}")


def _emulate_ln_fp32(x, shift, scale, one_pass):
    """The kernel's fp32 LayerNorm -> modulate on the CPU in its summation order (CPT channels per thread in order,
    then the 8 partial sums in order), with the centred two-pass variance or a one-pass E[x^2] - E[x]^2; fp16 out."""
    B, C, T = x.shape
    cpt = C // 8

    def ordered_sum(t):
        part = []
        for g in range(8):
            s = torch.zeros(B, T)
            for i in range(cpt):
                s = s + t[:, g * cpt + i]
            part.append(s)
        tot = torch.zeros(B, T)
        for s in part:
            tot = tot + s
        return tot[:, None, :]

    mean = ordered_sum(x) / C
    if one_pass:
        var = ordered_sum(x * x) / C - mean * mean
    else:
        d = x - mean
        var = ordered_sum(d * d) / C
    rstd = torch.rsqrt(var + LN_EPS)
    return (((x - mean) * rstd) * (1 + scale[:, :, None]) + shift[:, :, None]).half().double()


def test_ln_bound_fails_a_one_pass_variance():
    """The bound of (b) passes an emulation of the kernel's two-pass fp32 LayerNorm and fails the same with a one-pass
    variance at |mean| >> std."""
    B, C, T = 2, 256, 64
    gen = torch.Generator().manual_seed(3)
    x = torch.randn(B, C, T, generator=gen) * 0.5 + 300.0
    mod = torch.randn(B, 6 * C, generator=gen) * 0.5
    shift, scale = mod[:, :C], mod[:, C:2 * C]
    mask = torch.ones(B, T)
    _, ref, tol = _ln_ref(x, None, None, shift, scale, mask, False, False, False)
    ratio = {}
    for one_pass in (False, True):
        got = _emulate_ln_fp32(x, shift, scale, one_pass)
        r = (got - ref).abs() / tol
        ratio[one_pass] = float(torch.nan_to_num(r, nan=float("inf")).max())
    print(f"\n[bound] LayerNorm: error / bound  two-pass {ratio[False]:.3f}  one-pass {ratio[True]:.3f}")
    assert ratio[False] <= 1.0 < ratio[True], ratio


# ----------------------------------------------------------------------------------------------
# (c) the operand-writing conv epilogue
# ----------------------------------------------------------------------------------------------
OPERAND_MODES = ("none", "gate", "gelu", "lrelu", "wn")        # blk_mode 0..4 (4: hsv_conv1d_umma_wn_tail)
OPERAND_NT = (16, 32, 64, 128, 256)
# |d act / d pre| <= LIP: a conv error e moves the activation by at most LIP e (gate: tanh' <= 1 plus sigmoid' <= 1/4)
LIP = {"none": 1.0, "gate": 1.25, "gelu": 1.13, "lrelu": 1.0, "wn": 1.0}


def operand_key(blk_mode, n_tile):
    return f"operand-out:{OPERAND_MODES[blk_mode]}:n{n_tile}"


def _operand_shape(mode, nt):
    """(cin, cout, k, d) of a case: the front's shapes (WN in_layer 192 -> 384 k = 5 gate, FFN 192 -> 768 k = 5 gelu,
    1x1 res_skip WN tail of H = 192) and the DBlock / TTV ResBlock1 leaky_relu chains, widened where n_tile must
    divide the output."""
    if mode == "gate":
        return (192, 384, 5, 1) if 384 % nt == 0 else (256, 512, 5, 1)
    if mode == "gelu":
        return 192, 768, 5, 1
    if mode == "wn":
        return (192, 384, 1, 1) if 192 % nt == 0 else (256, 512, 1, 1)
    if mode == "lrelu":
        return (64, 128, 3, 1) if nt <= 128 else (256, 256, 3, 5)
    return 128, 256, 3, 2


OPERAND_MATRIX = [(mode, nt, *_operand_shape(mode, nt), L) for i, (mode, nt) in
                  enumerate((m, n) for m in OPERAND_MODES for n in OPERAND_NT)
                  for L in ((257, 383) if i % 2 else (255, 129))]          # L % 128 = 1 and 127
OPERAND_KEYS = frozenset(operand_key(OPERAND_MODES.index(c[0]), c[1]) for c in OPERAND_MATRIX)


@pytest.mark.gpu
@pytest.mark.parametrize("mode,nt,cin,cout,k,d,L", OPERAND_MATRIX)
def test_operand_out_vs_fp64(hsv, mode, nt, cin, cout, k, d, L):
    ops = hsv.ops
    ops.set_umma_debug(0)
    B = 3
    gen = torch.Generator().manual_seed(cin + cout + nt + L + OPERAND_MODES.index(mode))
    x = torch.randn(B, cin, L, generator=gen).to(DEV)
    w = (torch.randn(cout, cin, k, generator=gen) / (cin * k) ** 0.5).to(DEV)
    bias = torch.randn(cout, generator=gen).to(DEV)
    bc = torch.randn(B, 3, cout, generator=gen).to(DEV)[:, 1]            # strided rows
    mask = _prefix_mask([L, L - 37, 1], L, DEV)
    a = torch.zeros(ops.blk16_shape(B, cin, L), dtype=torch.float16, device=DEV)
    ops.pack_blk16(x, a)
    pre = F.conv1d(x.half().double(), w.half().double(), bias.double(), padding=(k - 1) // 2 * d, dilation=d)
    mk = mask.double()[:, None, :]
    H = cout // 2
    co = H if mode in ("gate", "wn") else cout
    got_blk = torch.zeros(ops.blk16_shape(B, co, L), dtype=torch.float16, device=DEV)
    if mode == "wn":
        xs = torch.randn(B, H, L, generator=gen).to(DEV)
        acc = torch.randn(B, H, L, generator=gen).to(DEV)
        xk, ak = xs.clone(), acc.clone()
        ops.conv1d_umma_wn_tail(a, ops.pack_conv_weight(w, nt), bias, xk, ak, mask, got_blk, nt)
        e = 2e-4 * max(1.0, float(pre.abs().max()))
        x_ref = (xs.double() + pre[:, :H]) * mk
        a_ref = acc.double() + pre[:, H:]
        assert float(((xk.double() - x_ref).abs() - e - _ulp32(x_ref)).max()) <= 0, float((xk.double() - x_ref).abs().max())
        assert float(((ak.double() - a_ref).abs() - e - _ulp32(a_ref)).max()) <= 0, float((ak.double() - a_ref).abs().max())
        ref = x_ref
    else:
        pre = pre + bc.double()[:, :, None]
        e = LIP[mode] * 2e-4 * max(1.0, float(pre.abs().max()))
        if mode == "gate":
            perm = ops.gate_permutation(cout, DEV)
            bcp = torch.empty(B, 3, cout, device=DEV)[:, 1]                  # strided rows, in the gate's order
            bcp.copy_(bc[:, perm])
            ops.conv1d_umma_blk(a, ops.pack_conv_weight(w[perm].contiguous(), nt), bias[perm].contiguous(), L, cin, cout,
                                k, d, nt, got_blk, ops.BLK_GATE, bc=bcp, mask=mask)
            ref = torch.tanh(pre[:, :H]) * torch.sigmoid(pre[:, H:])
        else:
            m = {"none": ops.BLK_NONE, "gelu": ops.BLK_GELU, "lrelu": ops.BLK_LRELU}[mode]
            ops.conv1d_umma_blk(a, ops.pack_conv_weight(w, nt), bias, L, cin, cout, k, d, nt, got_blk, m, bc=bc,
                                mask=mask)
            ref = {"none": lambda t: t, "gelu": lambda t: F.gelu(t, approximate="tanh"),
                   "lrelu": lambda t: F.leaky_relu(t, 0.1)}[mode](pre)
        ref = ref * mk
    rec = ops.last_launch_config(ops.LAUNCH_CONV)
    assert (rec["kind"], rec["n_tile"], rec["blk_mode"], rec["msub"], rec["warps"]) == (
        ops.CONV_OPERAND_OUT, nt, OPERAND_MODES.index(mode), 1, 4), rec
    got = ops.unpack_blk16(got_blk, co, L).double()
    err = (got - ref).abs()
    tol = _ulp16(ref) + e
    print(f"\n[parity] operand-out {mode} n{nt} L={L}: worst error / bound {float((err / tol).max()):.3f}")
    assert bool((err <= tol).all()), (float((err / tol).max()), e)
    assert bool((got * (1 - mk) == 0).all())
    raw = got_blk.view(-1, got_blk.shape[-2], got_blk.shape[-1])      # the next conv's zero padding rows
    assert float(raw[:, :ops.BLK_PAD].abs().max()) == 0.0 and float(raw[:, ops.BLK_PAD + L:].abs().max()) == 0.0


# ----------------------------------------------------------------------------------------------
# (d) census of the attention launches
# ----------------------------------------------------------------------------------------------
FRONT_VERIFIED = {f"mha:d{D}:{out}:{form}:kv{kv}:q{q}" for D in (96, 128) for out in ("f32", "blk16")
                  for form in ("none:post", "lens:pre", "vlen:post", "vlen:pre") for kv in (0, 1) for q in (0, 1)}
FRONT_VERIFIED |= {f"mha:d64:f32:none:post:kv{kv}:q{q}" for kv in (0, 1) for q in (0, 1)}


def _declared_front_keys():
    """The attention keys the cases of (a) assert (each case checks every key of its staging through the hook)."""
    keys = set()
    for D, out, form, pre in ATTN_CASES:
        keys |= {_mha_key_expected(D, out, form, pre, *_staging(T, qo, ko)) for T, _, qo, ko in _attn_runs(D)}
    return keys


def test_front_verified_set_is_covered_by_the_cases():
    missing = FRONT_VERIFIED - _declared_front_keys()
    assert not missing, sorted(missing)


_MHA_CALLS = {"hsv_mha", "hsv_mha_blk16", "hsv_mha_ragged"}


def _record_attention(hsv, monkeypatch, run):
    from megatts2_hierspeechpp_b200 import _lib
    ops = hsv.ops
    ops.set_mha_variant(0)
    seen, orig = {}, _lib.check
    last = [ops.last_launch_config(ops.LAUNCH_MHA)["launches"]]

    def recording_check(rc, what):
        orig(rc, what)
        if what in _MHA_CALLS:
            c = ops.last_launch_config(ops.LAUNCH_MHA)
            if c["launches"] != last[0]:
                last[0] = c["launches"]
                assert c["kernel"] == 0, c
                k = mha_key(c)
                seen[k] = seen.get(k, 0) + 1

    monkeypatch.setattr(_lib, "check", recording_check)
    with torch.no_grad():
        run()
    torch.cuda.synchronize()
    monkeypatch.setattr(_lib, "check", orig)
    return seen


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["synth", "tts"])
def test_census_workload_attention_verified(hsv, monkeypatch, workload):
    """One eager forward of a benchmark workload at B = 1 x 10 s: every attention launch runs the tensor-core kernel in
    a variant (a) verifies."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    import bench

    wl = bench.make_workload(argparse.Namespace(workload=workload, batch=1, seconds=10.0), 0)
    model = bench.build_model(wl, DEV)
    seen = _record_attention(hsv, monkeypatch, lambda: model(*[t.to(DEV) for t in wl["host_inputs"]]))
    print(f"\n[census] {wl['name']} attention: " + ", ".join(f"{k} x{n}" for k, n in sorted(seen.items())))
    assert seen, "no attention launch recorded"
    assert not sorted(set(seen) - FRONT_VERIFIED), sorted(set(seen) - FRONT_VERIFIED)


@pytest.mark.gpu
def test_census_per_item_synthesizer_attention_verified(hsv, monkeypatch):
    """A per-item synthesizer batch of 16 mixed source and prompt lengths, padded as runtime.ragged_prompt_batches
    pads them: every attention launch runs a variant (a) verifies."""
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
        vl = torch.tensor([lengths[i] for i in ids], dtype=torch.int32, device=DEV)
        tl = torch.tensor([prompts[i] for i in ids] * 2, dtype=torch.int32, device=DEV)
        s = _record_attention(hsv, monkeypatch, lambda: model.voice_conversion_noise_control(
            src.to(DEV), vl, mel.to(DEV), tl, f0.to(DEV), 0.333, False, 0.3, per_item=True))
        for k, c in s.items():
            seen[k] = seen.get(k, 0) + c
    print(f"\n[census] per-item synthesizer B={n} ({len(batches)} batches) attention: "
          + ", ".join(f"{k} x{c}" for k, c in sorted(seen.items())))
    assert seen, "no attention launch recorded"
    assert not sorted(set(seen) - FRONT_VERIFIED), sorted(set(seen) - FRONT_VERIFIED)
