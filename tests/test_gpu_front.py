"""The step before the vocoder (SURVEY.md §8f2) on the GPU: frame-rate kernels against torch, the drop-in modules against
the oracle restatement (oracle/functional_front.py, pinned bit-exact to the reference on CPU) run in strict fp32 on the
same device with the same CUDA generator seed (the noise draws happen in the same order and shapes)."""
import contextlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import MAX_ABS_TOL, SNR_DB_MIN
from oracle import closed_form as CF
from oracle import functional_front as FF
from oracle import synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@contextlib.contextmanager
def strict_fp32():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        yield
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _rel(got, ref):
    return float((got - ref).abs().max() / max(1e-6, float(ref.abs().max())))


def test_pack_act_modes(hsv):
    ops = hsv.ops
    g = torch.Generator().manual_seed(1)
    B, C, T = 2, 192, 77
    x = torch.randn(B, 2 * C, T, generator=g).to(DEV)
    bc = torch.randn(B, 2 * C, generator=g).to(DEV)
    mask = (torch.arange(T)[None, :] < torch.tensor([T, 50])[:, None]).float().to(DEV)
    buf = ops.blk16_buffer(B, C, T, DEV, slot=8)
    ops.pack_blk16_act(x, buf, C, ops.PACK_GATE, bcast=bc)
    a = x + bc.unsqueeze(-1)
    assert _rel(ops.unpack_blk16(buf, C, T), torch.tanh(a[:, :C]) * torch.sigmoid(a[:, C:])) <= 1e-3
    ops.pack_blk16_act(x, buf, C, ops.PACK_GELU, mask=mask)
    assert _rel(ops.unpack_blk16(buf, C, T), F.gelu(x[:, :C], approximate="tanh") * mask.unsqueeze(1)) <= 1e-3
    ops.pack_blk16_act(x, buf, C, ops.PACK_MISH, mask=mask, c_off=C)
    xm = x[:, C:]
    assert _rel(ops.unpack_blk16(buf, C, T), xm * torch.tanh(F.softplus(xm)) * mask.unsqueeze(1)) <= 1e-3
    ops.pack_blk16_act(x, buf, C, ops.PACK_MASK)
    assert _rel(ops.unpack_blk16(buf, C, T), x[:, :C]) <= 1e-3
    # arguments across softplus's threshold of 20 and saturated gate arguments, against fp64: within one fp16 spacing
    # of the value (2^-24 below the normal range) plus a few fp32 roundings of it
    xe = _edge_args(B, 2 * C, T, g).to(DEV)
    bz = torch.zeros(B, 2 * C, device=DEV)
    x64 = xe.double()
    for mode, ref in ((ops.PACK_GATE, torch.tanh(x64[:, :C]) * torch.sigmoid(x64[:, C:])),
                      (ops.PACK_MISH, x64[:, :C] * torch.tanh(F.softplus(x64[:, :C])))):
        ops.pack_blk16_act(xe, buf, C, mode, bcast=bz if mode == ops.PACK_GATE else None)
        got = ops.unpack_blk16(buf, C, T).double()
        ulp = torch.exp2(torch.floor(torch.log2(ref.abs().clamp_min(2.0 ** -14))) - 10)
        assert bool(((got - ref).abs() <= ulp + 1e-6 * ref.abs()).all()), (mode, float((got - ref).abs().max()))


def _edge_args(B, C, T, g):
    """Arguments in [-100, 100] with the exact values around softplus's threshold of 20 and deep saturation."""
    x = torch.rand(B, C, T, generator=g) * 200 - 100
    edges = torch.tensor([-100., -88., -40., -20.5, -20., -19.5, -1., 0., 1., 19.5, 19.999, 20., 20.001, 20.5, 40., 88.])
    x[..., :len(edges)] = edges
    x[:, ::2, len(edges):2 * len(edges)] = edges.flip(0)
    return x


@pytest.mark.parametrize("C", [192, 256])
def test_ln_mod(hsv, C):
    ops = hsv.ops
    g = torch.Generator().manual_seed(2)
    B, T = 2, 131
    x = (torch.randn(B, C, T, generator=g) * 3 + 1).to(DEV)
    mod = torch.randn(B, 6 * C, generator=g).to(DEV)
    mask = (torch.arange(T)[None, :] < torch.tensor([T, 90])[:, None]).float().to(DEV)
    buf = ops.blk16_buffer(B, C, T, DEV, slot=8)
    for premask in (False, True):
        ops.ln_mod_blk16(x, mod[:, C:2 * C], mod[:, 3 * C:4 * C], buf, 6 * C, mask, 1e-6, premask=premask)
        n = F.layer_norm(x.transpose(1, 2), (C,), None, None, 1e-6).transpose(1, 2)
        if premask:
            n = n * mask.unsqueeze(1)
        ref = n * (1 + mod[:, 3 * C:4 * C].unsqueeze(-1)) + mod[:, C:2 * C].unsqueeze(-1)
        assert _rel(ops.unpack_blk16(buf, C, T), ref) <= 1.5e-3


def test_gate_ln_mod_equals_two_launches(hsv):
    """x += gate * y * mask fused into the LayerNorm / modulate / pack launch == gate_add then ln_mod, bit for bit."""
    ops = hsv.ops
    g = torch.Generator().manual_seed(12)
    B, C, T = 2, 192, 131
    x = (torch.randn(B, C, T, generator=g) * 2).to(DEV)
    y = torch.randn(B, C, T, generator=g).to(DEV)
    mod = torch.randn(B, 3, 6 * C, generator=g).to(DEV)[:, 1]            # strided rows, as the batched adaLN gives them
    ms = mod.stride(0)
    mask = (torch.arange(T)[None, :] < torch.tensor([T, 90])[:, None]).float().to(DEV)
    a, b = ops.blk16_buffer(B, C, T, DEV, slot=8), ops.blk16_buffer(B, C, T, DEV, slot=9)
    for premask in (False, True):
        x1, x2 = x.clone(), x.clone()
        ops.frame_op(ops.OP_GATE_ADD, x1, y, mod[:, 2 * C:3 * C], mask, x1, None, B, C, T, cstride=ms)
        ops.ln_mod_blk16(x1, mod[:, :C], mod[:, C:2 * C], a, ms, mask, 1e-6, premask=premask)
        ops.gate_ln_mod_blk16(x2, y, mod[:, 2 * C:3 * C], mod[:, :C], mod[:, C:2 * C], b, ms, mask, 1e-6, premask=premask)
        assert torch.equal(x1, x2)
        assert torch.equal(ops.unpack_blk16(a, C, T), ops.unpack_blk16(b, C, T))


def test_frame_ops(hsv):
    ops = hsv.ops
    g = torch.Generator().manual_seed(3)
    B, C, T = 2, 96, 53
    mask = (torch.arange(T)[None, :] < torch.tensor([T, 31])[:, None]).float().to(DEV)
    mk = mask.unsqueeze(1)
    x = torch.randn(B, C, T, generator=g).to(DEV)
    rs = torch.randn(B, 2 * C, T, generator=g).to(DEV)
    o = torch.randn(B, C, T, generator=g).to(DEV)
    x1, o1 = x.clone(), o.clone()
    ops.frame_op(ops.OP_WN_RES, x1, rs, None, mask, x1, o1, B, C, T)
    assert torch.allclose(x1, (x + rs[:, :C]) * mk) and torch.allclose(o1, o + rs[:, C:])
    o2 = o.clone()
    ops.frame_op(ops.OP_WN_LAST, None, rs[:, :C].contiguous(), None, mask, None, o2, B, C, T)
    assert torch.allclose(o2, (o + rs[:, :C]) * mk)
    gate = torch.randn(B, 6 * C, generator=g).to(DEV)
    y = torch.randn(B, C, T, generator=g).to(DEV)
    x3 = x.clone()
    ops.frame_op(ops.OP_GATE_ADD, x3, y, gate[:, 2 * C:3 * C], mask, x3, None, B, C, T, cstride=6 * C)
    assert torch.allclose(x3, x + gate[:, 2 * C:3 * C].unsqueeze(-1) * y * mk, atol=1e-6)
    full = torch.randn(B, 2 * C, T, generator=g).to(DEV)
    f2 = full.clone()
    ops.frame_op(ops.OP_COUPLE, f2, y, None, mask, f2, None, B, C, T)
    assert torch.equal(f2[:, :C], full[:, :C]) and torch.allclose(f2[:, C:], (full[:, C:] - y) * mk)
    z = torch.empty(B, C, T, device=DEV)
    ops.frame_op(ops.OP_SAMPLE, full, y, None, mask, z, None, B, C, T, s=0.333)
    assert torch.allclose(z, (full[:, :C] + y * torch.exp(full[:, C:]) * 0.333) * mk, rtol=1e-5, atol=1e-6)
    out = torch.empty_like(x)
    ops.frame_op(ops.OP_GLU_RES, x, rs, None, mask, out, None, B, C, T)
    assert torch.allclose(out, (x + rs[:, :C] * torch.sigmoid(rs[:, C:])) * mk, atol=1e-6)
    ops.frame_op(ops.OP_MISH, x, None, None, mask, out, None, B, C, T)
    assert torch.allclose(out, x * torch.tanh(F.softplus(x)) * mk, atol=1e-6)
    xe = _edge_args(B, C, T, g).to(DEV)                 # across softplus's threshold of 20, against fp64
    ops.frame_op(ops.OP_MISH, xe, None, None, None, out, None, B, C, T)
    ref = xe.double() * torch.tanh(F.softplus(xe.double()))
    assert bool(((out.double() - ref).abs() <= 2e-6 * ref.abs() + 1e-37).all())       # + the fp32 subnormal range
    ys = torch.cat([_edge_args(B, C, T, g), _edge_args(B, C, T, g).flip(1)], 1).to(DEV)   # saturated sigmoid
    ops.frame_op(ops.OP_GLU_RES, x, ys, None, None, out, None, B, C, T)
    ref = x.double() + ys[:, :C].double() * torch.sigmoid(ys[:, C:].double())
    assert bool(((out.double() - ref).abs() <= 1e-6 * (x.double().abs() + ys[:, :C].double().abs())).all())
    ops.frame_op(ops.OP_FLIP, x, None, None, None, out, None, B, C, T)
    assert torch.equal(out, torch.flip(x, [1]))
    ops.frame_op(ops.OP_ADD, x, y, None, None, out, None, B, C, T)
    assert torch.equal(out, x + y)


@pytest.mark.parametrize("variant", [0, 1], ids=["tensor", "fp32"])
@pytest.mark.parametrize("D,T,masked", [(96, 500, False), (96, 37, False), (128, 150, True), (64, 70, True),
                                        (96, 500, True), (96, 1, False), (128, 16, False), (96, 68, True)])
def test_mha_vs_torch(hsv, D, T, masked, variant):
    """Both attention kernels against torch in strict fp32: the fp32 CUDA-core one to 2e-5; the mma.sync one (logits
    from hi/lo-split fp16 operands = fp32-level, P V in plain fp16 with fp32 accumulate) to 1e-3 of the peak -- the
    rounding the following proj conv's fp16 operand pack applies to the result anyway."""
    ops = hsv.ops
    ops.set_mha_variant(variant)
    try:
        _mha_case(hsv, D, T, masked, 1e-3 if variant == 0 else 2e-5)
    finally:
        ops.set_mha_variant(0)


def _mha_case(hsv, D, T, masked, tol):
    ops = hsv.ops
    g = torch.Generator().manual_seed(D + T)
    B, H = 2, 2
    C = H * D
    qkv = torch.randn(B, 3 * C, T, generator=g).to(DEV)
    lens = torch.tensor([T, max(1, T - 9)], dtype=torch.int32, device=DEV) if masked else None
    flat = qkv.view(-1)
    got = ops.mha(flat, flat[C * T:], flat[2 * C * T:], B, H, D, T, T, 3 * C * T, 3 * C * T, 3 * C * T, D ** -0.5,
                  prescale_q=masked, lens=lens)
    q, k, v = (qkv[:, i * C:(i + 1) * C].view(B, H, D, T).transpose(2, 3) for i in range(3))
    with strict_fp32():
        sc = torch.matmul(q * D ** -0.5, k.transpose(-2, -1)) if masked else torch.matmul(q, k.transpose(-2, -1)) * D ** -0.5
        if masked:
            m = (torch.arange(T, device=DEV)[None, :] < lens[:, None]).float()
            am = (m.unsqueeze(1) * m.unsqueeze(-1)).unsqueeze(1)
            sc = sc.masked_fill(am == 0, -1e4)
        ref = torch.matmul(sc.softmax(-1), v).transpose(2, 3).contiguous().view(B, C, T)
    err = _rel(got, ref)
    print(f"[parity] mha D={D} T={T} masked={masked}: rel={err:.2e}")
    assert err <= tol


def test_mha_blk16_output_equals_pack_of_fp32_output(hsv):
    """The attention kernel writing the proj conv's fp16 operand directly == its fp32 output packed afterwards."""
    ops = hsv.ops
    g = torch.Generator().manual_seed(4)
    for B, H, D, T in ((1, 2, 96, 500), (2, 2, 96, 77), (2, 2, 128, 41)):
        C = H * D
        qkv = torch.randn(B, 3 * C, T, generator=g).to(DEV)
        flat = qkv.view(-1)
        lens = torch.tensor([T, max(1, T - 5)][:B], dtype=torch.int32, device=DEV)
        args = (flat, flat[C * T:], flat[2 * C * T:], B, H, D, T, T, 3 * C * T, 3 * C * T, 3 * C * T, D ** -0.5, False)
        ref = ops.mha(*args, lens=lens)
        a, b = ops.blk16_buffer(B, C, T, DEV, slot=8), ops.blk16_buffer(B, C, T, DEV, slot=9)
        ops.mha(*args, lens=lens, out_blk=a)
        ops.pack_blk16(ref, b)
        assert torch.equal(ops.unpack_blk16(a, C, T), ops.unpack_blk16(b, C, T))


def test_wn_res_pack(hsv):
    ops = hsv.ops
    g = torch.Generator().manual_seed(6)
    B, C, T = 2, 192, 77
    x = torch.randn(B, C, T, generator=g).to(DEV)
    rs = torch.randn(B, 2 * C, T, generator=g).to(DEV)
    out = torch.randn(B, C, T, generator=g).to(DEV)
    mask = (torch.arange(T)[None, :] < torch.tensor([T, 50])[:, None]).float().to(DEV)
    x_ref = (x + rs[:, :C]) * mask.unsqueeze(1)
    out_ref = out + rs[:, C:]
    buf, ref_buf = ops.blk16_buffer(B, C, T, DEV, slot=8), ops.blk16_buffer(B, C, T, DEV, slot=9)
    ops.wn_res_pack(x, rs, mask, out, buf)
    assert torch.equal(x, x_ref) and torch.equal(out, out_ref)
    ops.pack_blk16(x_ref, ref_buf)
    assert torch.equal(ops.unpack_blk16(buf, C, T), ops.unpack_blk16(ref_buf, C, T))


def test_strided_conv_and_mean(hsv):
    ops = hsv.ops
    g = torch.Generator().manual_seed(5)
    x = torch.randn(2, 1, 403, generator=g).to(DEV)           # not a multiple of the stride
    w = torch.randn(192, 1, 9, generator=g).to(DEV)
    b = torch.randn(192, generator=g).to(DEV)
    ref = F.conv1d(x, w, b, stride=4, padding=4)
    assert torch.allclose(ops.conv1d_c1_strided(x, w, b, 4, 4), ref, atol=1e-5)
    h = torch.randn(2, 256, 77, generator=g).to(DEV)
    mask = (torch.arange(77)[None, :] < torch.tensor([77, 40])[:, None]).float().to(DEV)
    assert torch.allclose(ops.masked_mean(h, mask), h.sum(2) / mask.sum(1, keepdim=True), rtol=1e-5, atol=1e-6)


@pytest.fixture(scope="module")
def synthesizer(hsv):
    m = hsv.HierSpeechSynthesizer()
    m.load_state_dict(synth.synthesizer_sd(1234), strict=True)
    return m.to(DEV).eval()


def _inputs(T, T_mel, lens_mel):
    from megatts2_hierspeechpp_b200 import synthetic
    w2v, f0, mel = synthetic.synthesizer_inputs(T, T_mel, seed=1111)
    return (w2v.to(DEV), f0.to(DEV), mel.to(DEV), torch.LongTensor([T]).to(DEV), torch.LongTensor(lens_mel).to(DEV))


@pytest.mark.parametrize("T,T_mel,lens_mel", [(100, 150, [150, 150]), (37, 64, [64, 41])])
def test_front_modules_vs_oracle(hsv, synthesizer, T, T_mel, lens_mel):
    sd = {k: v.to(DEV) for k, v in synth.synthesizer_sd(1234).items()}
    w2v, f0, mel, ln, ln2 = _inputs(T, T_mel, lens_mel)
    with strict_fp32(), torch.no_grad():
        tm = torch.unsqueeze(FF.sequence_mask(ln2, mel.size(2)), 1).to(mel.dtype)
        g_ref = FF.style_encoder(sd, "emb_g.", mel, tm)
        g = synthesizer.emb_g(mel, tm)
        print(f"[parity] StyleEncoder g: rel={_rel(g, g_ref):.2e}")
        assert _rel(g, g_ref) <= 2e-3
        ym = torch.ones(1, 1, T, device=DEV)
        gi = g_ref[:1].unsqueeze(-1).contiguous()
        torch.manual_seed(5)
        z_ref, m_ref, l_ref = FF.posterior_sf_encoder(sd, "enc_p_l.", w2v, f0, ym, gi)
        torch.manual_seed(5)
        z, m, l = synthesizer.enc_p_l(w2v, f0, ym, g=gi)
        print(f"[parity] PosteriorSFEncoder z: rel={_rel(z, z_ref):.2e}  m: {_rel(m, m_ref):.2e}  logs: {_rel(l, l_ref):.2e}")
        assert _rel(z, z_ref) <= 2e-3 and _rel(m, m_ref) <= 2e-3 and _rel(l, l_ref) <= 2e-3
        f_ref = FF.coupling_block_reverse(sd, "flow_l.", z_ref, ym, gi)
        f = synthesizer.flow_l(z_ref, ym, g=gi, reverse=True)
        print(f"[parity] flow_l reverse: rel={_rel(f, f_ref):.2e}")
        assert _rel(f, f_ref) <= 2e-3


@pytest.mark.parametrize("T,T_mel,lens_mel", [(150, 150, [150, 150]), (500, 300, [300, 300])])
def test_voice_conversion_noise_control_vs_oracle(hsv, synthesizer, T, T_mel, lens_mel):
    """w2v + f0 + prompt mel -> 16 kHz waveform, everything on B200 kernels, vs the reference op sequence (config #2 at
    the SynthesizerTrn level for T = 500)."""
    sd = {k: v.to(DEV) for k, v in synth.synthesizer_sd(1234).items()}
    w2v, f0, mel, ln, ln2 = _inputs(T, T_mel, lens_mel)
    with strict_fp32(), torch.no_grad():
        torch.manual_seed(7)
        ref = FF.voice_conversion_noise_control(sd, w2v, ln, mel, ln2, f0, noise_scale=0.333, denoise_ratio=0.3)
        torch.manual_seed(7)
        got = synthesizer.voice_conversion_noise_control(w2v, ln, mel, ln2, f0, noise_scale=0.333, denoise_ratio=0.3)
    assert got.shape == (1, 1, 320 * T)
    ma, snr = CF.max_abs(ref.cpu().numpy(), got.cpu().numpy()), CF.snr_db(ref.cpu().numpy(), got.cpu().numpy())
    print(f"[parity] voice_conversion_noise_control T={T}: max_abs={ma:.3e} snr={snr:.1f} dB")
    assert ma <= MAX_ABS_TOL and snr >= SNR_DB_MIN
    # multi-stream mode (resblock streams, source_enc || filter_enc, pre-stage overlap) == single stream, bit for bit
    mods = [m for m in synthesizer.modules() if hasattr(m, "parallel_blocks")]
    try:
        for m in mods:
            m.parallel_blocks = True
        torch.manual_seed(7)
        with torch.no_grad():
            par = synthesizer.voice_conversion_noise_control(w2v, ln, mel, ln2, f0, noise_scale=0.333, denoise_ratio=0.3)
    finally:
        for m in mods:
            m.parallel_blocks = False
    assert torch.equal(par, got)
    # graph replay == eager (same seed before each)
    runner = hsv.CudaGraphRunner(lambda a, b, c: synthesizer.voice_conversion_noise_control(a, ln, c, ln2, b, 0.333, False, 0.3))
    torch.manual_seed(7)
    g1 = runner(w2v, f0, mel)
    assert g1.shape == got.shape and bool(torch.isfinite(g1).all())


@pytest.mark.parametrize("B,H,T", [(1, 192, 500), (2, 192, 77), (1, 512, 150)])
def test_wn_tail_epilogue_equals_conv_then_wn_res_pack(hsv, B, H, T):
    """The res_skip conv with the WN layer tail in its epilogue == the fp32 conv followed by wn_res_pack, bit for bit."""
    ops = hsv.ops
    g = torch.Generator().manual_seed(H + T)
    acts = torch.randn(B, H, T, generator=g).to(DEV)
    w = (torch.randn(2 * H, H, 1, generator=g) / H ** 0.5).to(DEV)
    bias = torch.randn(2 * H, generator=g).to(DEV)
    x = torch.randn(B, H, T, generator=g).to(DEV)
    out = torch.randn(B, H, T, generator=g).to(DEV)
    mask = (torch.arange(T)[None, :] < torch.tensor([T, max(1, T - 20)][:B])[:, None]).float().to(DEV)
    a = ops.blk16_buffer(B, H, T, DEV, slot=8)
    ops.pack_blk16(acts, a)
    nt = ops.pick_n_tile(2 * H, B * ((T + 127) // 128), H)
    assert H % nt == 0
    wp = ops.pack_conv_weight(w, nt)
    x1, o1, x2, o2 = x.clone(), out.clone(), x.clone(), out.clone()
    b1, b2 = ops.blk16_buffer(B, H, T, DEV, slot=9), ops.blk16_buffer(B, H, T, DEV, slot=10)
    rs = ops.conv1d_umma(a, wp, bias, T, H, 2 * H, 1, 1, nt)
    ops.wn_res_pack(x1, rs, mask, o1, b1)
    ops.conv1d_umma_wn_tail(a, wp, bias, x2, o2, mask, b2, nt)
    assert torch.equal(x1, x2) and torch.equal(o1, o2)
    assert torch.equal(ops.unpack_blk16(b1, H, T), ops.unpack_blk16(b2, H, T))
