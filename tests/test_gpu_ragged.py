"""Ragged batches on the GPU: utterances of different lengths padded into one batch, with per-utterance lengths.

Every item's valid region must equal, bit for bit (``torch.equal``), the same kernel / module on that item alone and
unpadded; everything past it must be exactly 0; input past an item's length is filled with NaN, so reading it would
show."""
import numpy as np
import pytest
import torch

from conftest import golden, golden_sd
from oracle import synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _nan_tail(x, lens):
    x = x.clone()
    for b, n in enumerate(lens):
        x[b, ..., n:] = float("nan")
    return x


def _lens(lens):
    return torch.tensor(lens, dtype=torch.int32, device=DEV)


def _check_items(out, ref_of, lens, scale=1):
    """out[b, ..., :scale*len] == ref_of(b) and out[b, ..., scale*len:] == 0 for every item."""
    for b, n in enumerate(lens):
        ref = ref_of(b)
        v = scale * n
        assert torch.equal(out[b:b + 1, ..., :v], ref), (b, n)
        assert bool((out[b, ..., v:] == 0).all()), (b, n)


# ---------------------------------------------------------------------------------------------- kernels
@pytest.fixture
def act_variant(hsv):
    yield hsv.ops.set_act_variant
    hsv.ops.set_act_variant(0)


@pytest.mark.parametrize("L", [600, 601])      # 601: L % 4 != 0, every tile staged without TMA
@pytest.mark.parametrize("C", [16, 64])
@pytest.mark.parametrize("R", [9, 17, 21, 25])
def test_act1d_ragged(hsv, act_variant, R, C, L):
    ops = hsv.ops
    act_variant(R << 8)
    lens = [1, 2, 5, 12, L - 1, L]
    B = len(lens)
    gen = torch.Generator().manual_seed(R * 1000 + C + L)
    x = _nan_tail(torch.randn(B, C, L, generator=gen).to(DEV), lens)
    al = (torch.rand(C, generator=gen) - 0.5).to(DEV)
    be = (torch.rand(C, generator=gen) - 0.5).to(DEV)
    vl = _lens(lens)
    # fp32 output
    out = ops.act1d(x, al, be, scale=0.5, valid_len=vl)
    assert ops.last_launch_config(ops.LAUNCH_ACT)["R"] == R
    _check_items(out, lambda b: ops.act1d(x[b:b + 1, :, :lens[b]].contiguous(), al, be, scale=0.5), lens)
    # fp16 operand output, into a buffer that already holds another full-length operand
    buf = torch.zeros(ops.blk16_shape(B, C, L), dtype=torch.float16, device=DEV)
    ops.pack_blk16(torch.randn(B, C, L, generator=gen).to(DEV) + 3.0, buf)
    ops.act1d_blk16(x, al, be, buf, scale=0.5, valid_len=vl)
    got = ops.unpack_blk16(buf, C, L)

    def ref_blk(b):
        n = lens[b]
        rb = torch.zeros(ops.blk16_shape(1, C, n), dtype=torch.float16, device=DEV)
        ops.act1d_blk16(x[b:b + 1, :, :n].contiguous(), al, be, rb, scale=0.5)
        return ops.unpack_blk16(rb, C, n)

    _check_items(got, ref_blk, lens)


@pytest.mark.parametrize("mode", ["one", "two", "three", "lrelu", "scale"])
def test_pack_blk16_ragged(hsv, mode):
    ops = hsv.ops
    B, C, L = 5, 32, 700
    lens = [700, 1, 3, 257, 699]
    gen = torch.Generator().manual_seed(3)
    n_add = {"two": 2, "three": 3}.get(mode, 1)
    xs = [_nan_tail(torch.randn(B, C, L, generator=gen).to(DEV), lens) for _ in range(n_add)]
    kw = {"lrelu": mode == "lrelu", "scale": 0.25 if mode == "scale" else 1.0}
    buf = torch.zeros(ops.blk16_shape(B, C, L), dtype=torch.float16, device=DEV)
    ops.pack_blk16(torch.ones(B, C, L, device=DEV), buf)
    ops.pack_blk16(xs if n_add > 1 else xs[0], buf, valid_len=_lens(lens), **kw)
    got = ops.unpack_blk16(buf, C, L)

    def ref(b):
        n = lens[b]
        rb = torch.zeros(ops.blk16_shape(1, C, n), dtype=torch.float16, device=DEV)
        item = [t[b:b + 1, :, :n].contiguous() for t in xs]
        ops.pack_blk16(item if n_add > 1 else item[0], rb, **kw)
        return ops.unpack_blk16(rb, C, n)

    _check_items(got, ref, lens)


@pytest.mark.parametrize("L", [1000, 1001])    # 1000: float4 kernel, 1001: scalar-staged kernel
def test_conv_post_ragged(hsv, L):
    ops = hsv.ops
    lens = [L, 1, 5, 8, 9, 13, 515, L - 1]     # <= 8: the warp-reduction order of a short sequence's own run
    B, C = len(lens), 32
    gen = torch.Generator().manual_seed(L)
    x = _nan_tail(torch.randn(B, C, L, generator=gen).to(DEV), lens)
    w = (torch.randn(1, C, 7, generator=gen) * 0.1).to(DEV)
    out = ops.conv1d_direct(x, w, None, pad=3, flags=ops.CONV_TANH, valid_len=_lens(lens))
    _check_items(out, lambda b: ops.conv1d_direct(x[b:b + 1, :, :lens[b]].contiguous(), w, None, pad=3,
                                                  flags=ops.CONV_TANH), lens)


@pytest.mark.parametrize("scale", [1.5, 3])
def test_sr_pre_interp_ragged(hsv, scale):
    ops = hsv.ops
    lens = [1000, 1, 7, 333, 999]
    B, C, L = len(lens), 8, 1000
    Lout = int(L * scale)
    louts = [int(n * scale) for n in lens]
    gen = torch.Generator().manual_seed(9)
    x = _nan_tail(torch.randn(B, 1, L, generator=gen).to(DEV), lens)
    w = torch.randn(C, 1, 7, generator=gen).to(DEV)
    bias = torch.randn(C, generator=gen).to(DEV)
    out = ops.sr_pre_interp(x, w, bias, Lout, valid_len=(_lens(lens), _lens(louts)))
    for b, n in enumerate(lens):
        ref = ops.sr_pre_interp(x[b:b + 1, :, :n].contiguous(), w, bias, louts[b])
        assert torch.equal(out[b:b + 1, :, :louts[b]], ref), b
        assert bool((out[b, :, louts[b]:] == 0).all()), b
    # per-item index tables: a ramp through a centre-tap filter reads back (1 - lam) * i0 + lam * i1 at Lin_b
    ramp = torch.arange(L, dtype=torch.float32, device=DEV).expand(B, 1, L).contiguous()
    delta = torch.zeros(1, 1, 7, device=DEV)
    delta[0, 0, 3] = 1.0
    got = ops.sr_pre_interp(ramp, delta, None, Lout, valid_len=(_lens(lens), _lens(louts)))
    for b, n in enumerate(lens):
        i0, i1, lam = (t.double() for t in ops.interp_linear_table(n, louts[b], DEV))
        want = ((1 - lam) * i0 + lam * i1).float()
        torch.testing.assert_close(got[b, 0, :louts[b]], want, rtol=0, atol=2e-3 * max(n, 1) ** 0.5)


# ---------------------------------------------------------------------------------------------- modules
@pytest.fixture(scope="module")
def vocoder(hsv):
    m = hsv.Vocoder()
    m.load_state_dict(synth.vocoder_sd(1234), strict=True)
    return m.to(DEV).eval()


@pytest.mark.parametrize("parallel", [False, True])
def test_vocoder_ragged_items_equal_their_own_runs(vocoder, parallel):
    lens = [500, 1, 2, 37, 499, 250]
    B, T = len(lens), max(lens)
    z, g = synth.vocoder_inputs(B, T, seed=21)
    z, g = _nan_tail(z.to(DEV), lens), g.to(DEV)
    vocoder.dec.parallel_blocks = vocoder.sn.parallel_blocks = parallel
    try:
        with torch.no_grad():
            out = vocoder(z, g, lengths=torch.tensor(lens, device=DEV))      # int64 device tensor
            assert out.shape == (B, 1, 320 * T)
            _check_items(out, lambda b: vocoder(z[b:b + 1, :, :lens[b]].contiguous(), g[b:b + 1]), lens, scale=320)
            assert torch.equal(vocoder(z, g, lengths=lens), out)              # host sequence
    finally:
        vocoder.dec.parallel_blocks = vocoder.sn.parallel_blocks = False


def test_full_lengths_equal_the_unragged_path(vocoder):
    z, g = synth.vocoder_inputs(3, 40, seed=5)
    z, g = z.to(DEV), g.to(DEV)
    with torch.no_grad():
        assert torch.equal(vocoder(z, g, lengths=[40] * 3), vocoder(z, g))


@pytest.mark.parametrize("which", [24, 48])
def test_speechsr_ragged_items_equal_their_own_runs(hsv, which):
    sd = golden_sd(f"speechsr{which}_state.npz")
    m = (hsv.SpeechSR24 if which == 24 else hsv.SpeechSR48)(100, 40, **hsv.SR_CFG)
    m.load_state_dict(sd, strict=True)
    m.to(DEV).eval()
    wav = torch.from_numpy(golden("speechsr24_example.npz")["x_int16"].astype(np.float32) / 32768.0).to(DEV)
    lens = [48000, 1, 7, 16001, 3333]
    L = max(lens)
    x = torch.stack([torch.roll(wav[:L], 1000 * b) for b in range(len(lens))]).view(len(lens), 1, L)
    x = _nan_tail(x, lens)
    s = 1.5 if which == 24 else 3
    with torch.no_grad():
        out = m(x, lengths=_lens(lens))
        assert out.shape[-1] == int(L * s)
        for b, n in enumerate(lens):
            v = int(n * s)
            assert torch.equal(out[b:b + 1, :, :v], m(x[b:b + 1, :, :n].contiguous())), (which, n)
            assert bool((out[b, :, v:] == 0).all())
        assert torch.equal(m(x[:1], lengths=[L]), m(x[:1]))


def test_vocoder_sr_pcm16_ragged(hsv):
    chain = hsv.VocoderSR(24)
    sdc = {"vocoder." + k: v for k, v in synth.vocoder_sd(1234).items()}
    sdc.update({"sr." + k: v for k, v in golden_sd("speechsr24_state.npz").items()})
    chain.load_state_dict(sdc, strict=True)
    chain.to(DEV).eval()
    lens = [50, 20, 7]
    z, g = synth.vocoder_inputs(3, 50, seed=77)
    z, g = _nan_tail(z.to(DEV), lens), g.to(DEV)
    with torch.no_grad():
        pcm = chain(z, g, pcm16=True, lengths=_lens(lens))
        assert pcm.dtype == torch.int16 and pcm.shape == (3, 1, 480 * 50)
        # zero tails leave each row's peak (and so its PCM scale) unchanged
        _check_items(pcm, lambda b: chain(z[b:b + 1, :, :lens[b]].contiguous(), g[b:b + 1], pcm16=True), lens,
                     scale=480)


@pytest.mark.parametrize("parallel", [False, True])
def test_one_graph_serves_every_length_mix(hsv, vocoder, parallel):
    B, T = 3, 60
    z, g = synth.vocoder_inputs(B, T, seed=8)
    z, g = z.to(DEV), g.to(DEV)
    vocoder.dec.parallel_blocks = vocoder.sn.parallel_blocks = parallel
    try:
        runner = hsv.CudaGraphRunner(vocoder)
        with torch.no_grad():
            for lens in ([60, 13, 41], [7, 60, 59]):
                zz = _nan_tail(z, lens)
                got = runner(zz, g, _lens(lens)).clone()
                assert torch.equal(got, vocoder(zz, g, lengths=lens))
                assert torch.equal(got[2:3, :, :320 * lens[2]], vocoder(zz[2:3, :, :lens[2]].contiguous(), g[2:3]))
        assert runner.captures == 1
    finally:
        vocoder.dec.parallel_blocks = vocoder.sn.parallel_blocks = False


def test_bad_lengths_are_rejected(hsv, vocoder):
    z, g = synth.vocoder_inputs(2, 10, seed=1)
    z, g = z.to(DEV), g.to(DEV)
    bad = [[10], [10, 11], [0, 10], [10, -1], torch.tensor([10, 10]),             # wrong count / range / CPU
           torch.tensor([[10, 10]], device=DEV), torch.tensor([10.0, 10.0], device=DEV)]
    for lens in bad:
        with pytest.raises(ValueError):
            vocoder(z, g, lengths=lens)


def test_fused_half_layer_takes_no_lengths(hsv):
    from megatts2_hierspeechpp_b200 import modules as M
    gen = torch.Generator().manual_seed(11)
    sd = {}
    synth._amp_block(sd, "", gen, 16, 7)
    blk = hsv.AMPBlock1(16, 7, (1, 3, 5))
    blk.load_state_dict(sd, strict=True)
    blk.to(DEV)
    x = torch.randn(2, 16, 100, device=DEV)
    old = M.FUSE_MAX_CHANNELS[0]
    M.FUSE_MAX_CHANNELS[0] = 64
    try:
        with pytest.raises(NotImplementedError):
            blk.run(x, valid_len=_lens([100, 50]))
    finally:
        M.FUSE_MAX_CHANNELS[0] = old
