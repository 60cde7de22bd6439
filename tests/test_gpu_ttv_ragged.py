"""Per-item batches of the text-to-vec tail on the GPU: utterances of different lengths padded into one batch.

Every item must equal, bit for bit (``torch.equal``), the same kernel / module / chain on that item alone and unpadded;
everything past it must be exactly 0.  Input past an item's length is filled with large finite garbage, so reading it
would show."""
import pytest
import torch

from oracle import closed_form as CF
from oracle import functional_ttv as FT
from oracle import synth
from test_gpu_front import _rel, strict_fp32
from test_gpu_synth_ragged import _check_items, _garbage_tail, _lens, _own_noise, _packed
from test_gpu_variants import _CONV_CALLS, VERIFIED, act_key, conv_key

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


# ---------------------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("L", [131, 1000])
def test_strided_operand_split_k_k7_equals_dense(hsv, L):
    """PitchPredictor.conv_pre per item: k = 7 split-K passes reading channel ranges of ONE packed [B, 1024, L] buffer
    (the halo rows of every chunk) == the same passes on each item's dense copy, and on the item alone at its length."""
    ops = hsv.ops
    C, cout, k = 1024, 256, 7
    lens = [L, L - 3, 40, 1]
    B, per = len(lens), C // 2
    buf = _packed(ops, C, L, B, seed=L, lens=lens)
    nchunk = buf.shape[1] // 2
    gen = torch.Generator().manual_seed(L + 1)
    ws = [(torch.randn(cout, per, k, generator=gen) * 0.02).to(DEV) for _ in range(2)]
    bias = torch.randn(cout, generator=gen).to(DEV)
    nt = ops.pick_n_tile(cout)
    wp = [ops.pack_conv_weight(w, nt) for w in ws]

    def split_k(src, n):
        out = None
        for i in range(2):
            out = ops.conv1d_umma(src[:, i * nchunk:(i + 1) * nchunk], wp[i], bias if i == 0 else None, n, per, cout, k,
                                  1, nt, residual=out)
        return out

    got = split_k(buf, L)
    x = ops.unpack_blk16(buf, C, L)
    for b, n in enumerate(lens):
        assert torch.equal(got[b:b + 1], split_k(buf[b:b + 1].contiguous(), L)), b
        one = torch.zeros(ops.blk16_shape(1, C, n), dtype=torch.float16, device=DEV)
        ops.pack_blk16(x[b:b + 1, :, :n].contiguous(), one)
        assert torch.equal(got[b:b + 1, :, :n], split_k(one, n)), (b, n)


def test_conv_post_ragged_cin64_lrelu001(hsv):
    """PitchPredictor.conv_post (64 -> 1, k 7, leaky_relu(0.01) on the input) per item: items of 4n <= 8 samples take
    the row-dot order of their own short run, longer ones the thin kernel's."""
    ops = hsv.ops
    frames = [50, 3, 2, 1]
    lens = [4 * n for n in frames]
    B, L = len(lens), max(lens)
    gen = torch.Generator().manual_seed(64)
    x = _garbage_tail(torch.randn(B, 64, L, generator=gen).to(DEV), lens)
    w = (torch.randn(1, 64, 7, generator=gen) * 0.05).to(DEV)
    out = ops.conv1d_direct(x, w, None, pad=3, flags=ops.CONV_LRELU001_IN, valid_len=_lens(lens))
    _check_items(out, lambda b: ops.conv1d_direct(x[b:b + 1, :, :lens[b]].contiguous(), w, None, pad=3,
                                                  flags=ops.CONV_LRELU001_IN), lens)


# ---------------------------------------------------------------------------------------------- modules
@pytest.fixture(scope="module")
def tail(hsv):
    m = hsv.TTVTail()
    m.load_state_dict(synth.ttv_tail_sd(3456), strict=True)
    return m.to(DEV).eval()


def _inputs(lens, T, seed):
    z, _, g = synth.ttv_tail_inputs(len(lens), T, seed=seed)
    return _garbage_tail(z.to(DEV), lens, seed=seed), g.to(DEV)


def _own(tail, z, g, b, n):
    """The unbatched call on item b: batch 1, unpadded, y_mask = ones."""
    return tail(z[b:b + 1, :, :n].contiguous(), torch.ones(1, 1, n, device=DEV), g[b:b + 1].contiguous())


def _check_tail(tail, z, g, lens):
    with torch.no_grad():
        w2v, pitch = tail(z, None, g, lengths=_lens(lens))
        assert w2v.shape == (len(lens), 1024, z.shape[-1]) and pitch.shape == (len(lens), 1, 4 * z.shape[-1])
        for b, n in enumerate(lens):
            w_o, p_o = _own(tail, z, g, b, n)
            assert torch.equal(w2v[b:b + 1, :, :n], w_o) and bool((w2v[b, :, n:] == 0).all()), (b, n)
            assert torch.equal(pitch[b:b + 1, :, :4 * n], p_o) and bool((pitch[b, :, 4 * n:] == 0).all()), (b, n)
    return w2v, pitch


@pytest.fixture(params=[True, False], ids=["parallel", "serial"])
def parallel_blocks(request, tail):
    old = type(tail.pp).parallel_blocks
    type(tail.pp).parallel_blocks = request.param
    yield request.param
    type(tail.pp).parallel_blocks = old


def test_batch_of_one_at_full_length(tail, parallel_blocks):
    T = 200
    z, g = _inputs([T], T, seed=21)
    w2v, pitch = _check_tail(tail, z, g, [T])
    with torch.no_grad():
        w_n, p_n = tail(z, torch.ones(1, 1, T, device=DEV), g)
        w_h, p_h = tail(z, None, g, lengths=[T])                       # host sequence
    assert torch.equal(w2v, w_n) and torch.equal(pitch, p_n)
    assert torch.equal(w2v, w_h) and torch.equal(pitch, p_h)


def test_items_equal_their_own_runs(tail, parallel_blocks):
    lens = [333, 300, 129, 1]
    z, g = _inputs(lens, max(lens), seed=22)
    w2v, pitch = _check_tail(tail, z, g, lens)
    zero = z.clone()
    for b, n in enumerate(lens):
        zero[b, :, n:] = 0
    with torch.no_grad():
        w0, p0 = tail(zero, torch.ones(len(lens), 1, max(lens), device=DEV), g, lengths=_lens(lens))  # y_mask not read
    assert torch.equal(w0, w2v) and torch.equal(p0, pitch)


def test_sixteen_random_lengths(tail):
    T = 400
    lens = torch.randint(1, T + 1, (16,), generator=torch.Generator().manual_seed(16)).tolist()
    lens[3] = T
    z, g = _inputs(lens, T, seed=23)
    _check_tail(tail, z, g, lens)


def test_stage_sum_chained_in_the_batch_separate_alone(hsv, tail):
    """B = 16, T = 2100: the first stage's [16, 128, 4200] tensor is above SEPARATE_MAX_ELEMS, so the batch sums its
    resblocks in the conv epilogues while each item's own run takes them as separate tensors into the next pack."""
    from megatts2_hierspeechpp_b200 import modules
    T = 2100
    assert 16 * 128 * 2 * T > modules.SEPARATE_MAX_ELEMS[0] >= 128 * 2 * T
    lens = [T, 2099, 1999, 1500, 1024, 1023, 800, 640, 513, 512, 300, 129, 128, 50, 2, 1]
    z, g = _inputs(lens, T, seed=24)
    _check_tail(tail, z, g, lens)


def test_modules_alone(tail):
    """W2VDecoder and PitchPredictor each on their own: garbage in the padding of their input is never read."""
    lens = [250, 199, 64, 3]
    B, T = len(lens), max(lens)
    z, g = _inputs(lens, T, seed=25)
    x = _garbage_tail(torch.randn(B, 1024, T, generator=torch.Generator().manual_seed(26)).to(DEV), lens, seed=9)
    vl = _lens(lens)
    with torch.no_grad():
        w2v = tail.w2v_decoder(z, None, g=g, lengths=vl)
        pitch = tail.pp(x, g, lengths=vl)
        for b, n in enumerate(lens):
            one, gb = torch.ones(1, 1, n, device=DEV), g[b:b + 1].contiguous()
            assert torch.equal(w2v[b:b + 1, :, :n], tail.w2v_decoder(z[b:b + 1, :, :n].contiguous(), one, g=gb)), b
            assert bool((w2v[b, :, n:] == 0).all()), b
            assert torch.equal(pitch[b:b + 1, :, :4 * n], tail.pp(x[b:b + 1, :, :n].contiguous(), gb)), b
            assert bool((pitch[b, :, 4 * n:] == 0).all()), b


def test_item_of_a_batch_vs_oracle(tail):
    lens = [160, 97, 31]
    z, g = _inputs(lens, max(lens), seed=27)
    sd = {k: v.to(DEV) for k, v in synth.ttv_tail_sd(3456).items()}
    b, n = 1, lens[1]
    with strict_fp32(), torch.no_grad():
        w2v, pitch = tail(z, None, g, lengths=_lens(lens))
        w_ref, p_ref = FT.ttv_tail(sd, z[b:b + 1, :, :n].contiguous(), torch.ones(1, 1, n, device=DEV),
                                   g[b:b + 1].contiguous())
    w, p = w2v[b:b + 1, :, :n], pitch[b:b + 1, :, :4 * n]
    snr_w = CF.snr_db(w_ref.cpu().numpy(), w.cpu().numpy())
    snr_p = CF.snr_db(p_ref.cpu().numpy(), p.cpu().numpy())
    print(f"[parity] per-item W2VDecoder n={n}: rel={_rel(w, w_ref):.2e} snr={snr_w:.1f} dB   PitchPredictor: "
          f"rel={_rel(p, p_ref):.2e} snr={snr_p:.1f} dB")
    assert _rel(w, w_ref) <= 2e-3 and snr_w >= 55.0
    assert _rel(p, p_ref) <= 2e-3 and snr_p >= 55.0


# ---------------------------------------------------------------------------------------------- the TTS chain
@pytest.fixture(scope="module")
def synthesizer(hsv):
    m = hsv.HierSpeechSynthesizer()
    m.load_state_dict(synth.synthesizer_sd(1234), strict=True)
    return m.to(DEV).eval()


def _prompts(prompts, seed):
    mels = [synth.synthesizer_inputs(1, p, seed=seed + i)[2].to(DEV) for i, p in enumerate(prompts)]
    B, Tm = len(prompts), max(prompts)
    mel = torch.zeros(2 * B, 80, Tm, device=DEV)
    for b, (m, p) in enumerate(zip(mels, prompts)):
        mel[b, :, :p], mel[B + b, :, :p] = m[0], m[1]
    return mels, _garbage_tail(mel, prompts + prompts, seed=seed)


def _chain(tail, synthesizer, z, g, vl, mel, tl, eps):
    w2v, pitch = tail(z, None, g, lengths=vl)
    return synthesizer.voice_conversion_noise_control(w2v, vl, mel, tl, pitch, 0.333, False, 0.3, per_item=True,
                                                      eps=eps)


def test_tts_chain_items_equal_their_own_calls(tail, synthesizer):
    lens, prompts = [300, 211, 64, 5], [150, 217, 101, 64]
    B, T = len(lens), max(lens)
    z, g = _inputs(lens, T, seed=30)
    mels, mel = _prompts(prompts, seed=31)
    eps = torch.zeros(B, 192, T, device=DEV)
    for b, n in enumerate(lens):
        eps[b, :, :n] = _own_noise(200 + b, n, 2)[-1][0]
    eps = _garbage_tail(eps, lens, seed=32)
    with torch.no_grad():
        out = _chain(tail, synthesizer, z, g, _lens(lens), mel, _lens(prompts + prompts), eps)
        assert out.shape == (B, 1, 320 * T)

        def own(b):
            n, p = lens[b], prompts[b]
            w2v, pitch = _own(tail, z, g, b, n)
            torch.manual_seed(200 + b)
            return synthesizer.voice_conversion_noise_control(w2v, torch.LongTensor([n]).to(DEV), mels[b],
                                                              torch.LongTensor([p, p]).to(DEV), pitch, 0.333, False, 0.3)

        _check_items(out, own, lens, scale=320)


def test_one_graph_serves_every_length_mix(hsv, tail, synthesizer):
    B, T, Tm = 3, 120, 100
    z, g = _inputs([T] * B, T, seed=40)
    _, mel = _prompts([Tm] * B, seed=41)
    eps = torch.randn(B, 192, T, generator=torch.Generator().manual_seed(42)).to(DEV)

    def call(zz, gg, vl, m, tl, e):
        return _chain(tail, synthesizer, zz, gg, vl, m, tl, e)

    runner = hsv.CudaGraphRunner(call)
    with torch.no_grad():
        for lens, prompts in (([120, 13, 77], [100, 51, 9]), ([7, 120, 119], [99, 100, 64])):
            zz, m = _garbage_tail(z, lens, seed=43), _garbage_tail(mel, prompts + prompts, seed=44)
            vl, tl = _lens(lens), _lens(prompts + prompts)
            got = runner(zz, g, vl, m, tl, eps).clone()
            assert torch.equal(got, call(zz, g, vl, m, tl, eps))
            assert all(bool((got[b, :, 320 * n:] == 0).all()) for b, n in enumerate(lens))
    assert runner.captures == 1


def test_census_per_item_variants_verified(hsv, tail, synthesizer, monkeypatch):
    """Every conv / activation variant the per-item TTS chain launches is one tests/test_gpu_variants.py verifies."""
    from megatts2_hierspeechpp_b200 import _lib
    ops = hsv.ops
    ops.set_umma_debug(0)
    ops.set_act_variant(0)
    calls = set(_CONV_CALLS) | {"hsv_conv1d_umma_astride"}
    seen, orig = {}, _lib.check
    last = {f: ops.last_launch_config(f)["launches"] for f in (ops.LAUNCH_CONV, ops.LAUNCH_ACT)}

    def recording_check(rc, what):
        orig(rc, what)
        fam = ops.LAUNCH_CONV if what in calls else (ops.LAUNCH_ACT if what == "hsv_act1d_snakebeta" else None)
        if fam is not None:
            c = ops.last_launch_config(fam)
            if c["launches"] != last[fam]:
                last[fam] = c["launches"]
                k = conv_key(c) if fam == ops.LAUNCH_CONV else act_key(c)
                seen[k] = seen.get(k, 0) + 1

    # one micro-batch of the benchmark's size: 16 items up to 1000 frames
    lens = torch.randint(100, 1001, (16,), generator=torch.Generator().manual_seed(50)).tolist()
    lens[0] = T = 1000
    prompts = [300] * 16
    z, g = _inputs(lens, T, seed=51)
    _, mel = _prompts(prompts, seed=52)
    with torch.no_grad():
        _chain(tail, synthesizer, z, g, _lens(lens), mel, _lens(prompts + prompts), None)     # weights folded, packed
        torch.cuda.synchronize()
        monkeypatch.setattr(_lib, "check", recording_check)
        _chain(tail, synthesizer, z, g, _lens(lens), mel, _lens(prompts + prompts), None)
    torch.cuda.synchronize()
    monkeypatch.setattr(_lib, "check", orig)
    print("\n[census] per-item TTS chain: " + ", ".join(f"{k} x{n}" for k, n in sorted(seen.items())))
    assert seen
    assert not sorted(set(seen) - VERIFIED)
