"""Per-item batches of the synthesizer front on the GPU: utterances of different lengths padded into one batch.

Every item must equal, bit for bit (``torch.equal``), the same kernel / module / method on that item alone and unpadded;
everything past it must be exactly 0.  Input past an item's length is filled with large finite garbage, so reading it
would show."""
import pytest
import torch

from oracle import synth
from test_gpu_variants import _CONV_CALLS, VERIFIED, act_key, conv_key

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GARBAGE = 3.0e4


def _lens(lens):
    return torch.tensor(lens, dtype=torch.int32, device=DEV)


def _garbage_tail(x, lens, scale=1, seed=0):
    """x with x[b, ..., scale * lens[b]:] replaced by +-GARBAGE-sized finite values."""
    x = x.clone()
    gen = torch.Generator(device=x.device).manual_seed(seed)
    junk = (torch.rand(x.shape, generator=gen, device=x.device) - 0.5) * (2 * GARBAGE)
    for b, n in enumerate(lens):
        x[b, ..., scale * n:] = junk[b, ..., scale * n:]
    return x


def _check_items(out, ref_of, lens, scale=1):
    for b, n in enumerate(lens):
        v = scale * n
        assert torch.equal(out[b:b + 1, ..., :v], ref_of(b)), (b, n)
        assert bool((out[b, ..., v:] == 0).all()), (b, n)


# ---------------------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("out_blk", [False, True])
@pytest.mark.parametrize("D", [96, 128])
@pytest.mark.parametrize("T", [150, 157])           # 157: T % 4 != 0, every key tile staged with 4-byte copies
def test_mha_valid_len_items_equal_their_own_launch(hsv, T, D, out_blk):
    ops = hsv.ops
    heads, lens = 2, [T, T - 1, 17, 1]
    B, C = len(lens), 2 * D
    gen = torch.Generator().manual_seed(T + D)
    q, k, v = (_garbage_tail(torch.randn(B, C, T, generator=gen).to(DEV), lens, seed=i) for i in range(3))
    scale = D ** -0.5

    def run(qq, kk, vv, n, Bn, vl=None):
        if out_blk:
            buf = torch.zeros(ops.blk16_shape(Bn, C, n), dtype=torch.float16, device=DEV)
            if vl is not None:
                ops.pack_blk16(torch.full((Bn, C, n), 7.0, device=DEV), buf)     # rows past an item must be rewritten
            ops.mha(qq, kk, vv, Bn, heads, D, n, n, C * n, C * n, C * n, scale, False, out_blk=buf, valid_len=vl)
            return ops.unpack_blk16(buf, C, n)
        return ops.mha(qq, kk, vv, Bn, heads, D, n, n, C * n, C * n, C * n, scale, False, valid_len=vl)

    out = run(q, k, v, T, B, _lens(lens))
    _check_items(out, lambda b: run(*(t[b:b + 1, :, :lens[b]].contiguous() for t in (q, k, v)), lens[b], 1), lens)


def test_mha_valid_len_is_rejected_where_it_does_not_apply(hsv):
    ops = hsv.ops
    q = torch.randn(2, 192, 20, device=DEV)
    with pytest.raises(ValueError):
        ops.mha(q, q, q, 2, 2, 96, 20, 20, 0, 0, 0, 0.1, False, lens=_lens([20, 9]), valid_len=_lens([20, 9]))
    from megatts2_hierspeechpp_b200._lib import HsvError
    ops.set_mha_variant(1)
    try:
        with pytest.raises(HsvError):
            ops.mha(q, q, q, 2, 2, 96, 20, 20, 192 * 20, 192 * 20, 192 * 20, 0.1, False, valid_len=_lens([20, 9]))
    finally:
        ops.set_mha_variant(0)


def _packed(ops, C, L, B, seed, lens=None):
    x = torch.randn(B, C, L, generator=torch.Generator().manual_seed(seed)).to(DEV)
    if lens is not None:
        for b, n in enumerate(lens):
            x[b, :, n:] = 0
    buf = torch.zeros(ops.blk16_shape(B, C, L), dtype=torch.float16, device=DEV)
    ops.pack_blk16(x, buf)
    return buf


@pytest.mark.parametrize("C,L", [(768, 300), (1024, 131)])
def test_strided_operand_split_k_equals_dense_slices(hsv, C, L):
    """Split-K passes reading channel ranges of ONE packed [B] buffer == per-item launches on dense copies."""
    ops = hsv.ops
    B, cout = 3, 192
    per = C // 2
    buf = _packed(ops, C, L, B, seed=C)
    nchunk = buf.shape[1] // 2
    gen = torch.Generator().manual_seed(C + 1)
    ws = [(torch.randn(cout, per, 1, generator=gen) * 0.05).to(DEV) for _ in range(2)]
    bias = torch.randn(cout, generator=gen).to(DEV)
    nt = ops.pick_n_tile(cout)
    wp = [ops.pack_conv_weight(w, nt) for w in ws]

    def split_k(src):
        out = None
        for i in range(2):
            out = ops.conv1d_umma(src[:, i * nchunk:(i + 1) * nchunk], wp[i], bias if i == 0 else None, L, per, cout, 1,
                                  1, nt, residual=out)
        return out

    got = split_k(buf)
    for b in range(B):
        assert torch.equal(got[b:b + 1], split_k(buf[b:b + 1].contiguous())), b
    with pytest.raises(ValueError):          # a view that is not a chunk range of one buffer
        ops.conv1d_umma(buf[:, :, ::2], wp[0], None, L, per, cout, 1, 1, nt)


@pytest.mark.parametrize("cin,cout,k", [(192, 768, 5), (256, 512, 5), (192, 576, 1), (512, 192, 1)])
def test_conv_result_does_not_depend_on_the_tiles(hsv, cin, cout, k):
    """A per-item batch launches its convs with the tiles ``_row_tiles(B, T)`` picks, an item's own run with those of
    (1, len): the output must not depend on the output-channel tile or the row tiling (batch, length, sub-tiles)."""
    ops = hsv.ops
    lens = [300, 173, 17]
    B, L = len(lens), 300
    gen = torch.Generator().manual_seed(cin + cout + k)
    w = (torch.randn(cout, cin, k, generator=gen) * 0.05).to(DEV)
    bias = torch.randn(cout, generator=gen).to(DEV)
    buf = _packed(ops, cin, L, B, seed=k, lens=lens)
    tiles = [n for n in (16, 32, 64, 128, 256) if cout % n == 0]
    outs = {nt: ops.conv1d_umma(buf, ops.pack_conv_weight(w, nt), bias, L, cin, cout, k, 1, nt) for nt in tiles}
    ref = outs[tiles[0]]
    for nt, o in outs.items():
        assert torch.equal(o, ref), nt
    x = ops.unpack_blk16(buf, cin, L)
    for b, n in enumerate(lens):
        one = torch.zeros(ops.blk16_shape(1, cin, n), dtype=torch.float16, device=DEV)
        ops.pack_blk16(x[b:b + 1, :, :n].contiguous(), one)
        for nt in tiles:
            o = ops.conv1d_umma(one, ops.pack_conv_weight(w, nt), bias, n, cin, cout, k, 1, nt)
            assert torch.equal(o, ref[b:b + 1, :, :n]), (b, nt)


def test_strided_f0_conv_ragged(hsv):
    ops = hsv.ops
    lens = [100, 99, 7, 1]
    B, T = len(lens), 100
    gen = torch.Generator().manual_seed(4)
    x = _garbage_tail(torch.randn(B, 1, 4 * T, generator=gen).to(DEV), lens, scale=4)
    w = torch.randn(192, 1, 9, generator=gen).to(DEV)
    bias = torch.randn(192, generator=gen).to(DEV)
    vl = _lens(lens)
    mask = (torch.arange(T, device=DEV)[None, :] < vl[:, None]).float()
    out = ops.conv1d_c1_strided(x, w, bias, 4, 4, mask, valid_len=vl)
    _check_items(out, lambda b: ops.conv1d_c1_strided(x[b:b + 1, :, :4 * lens[b]].contiguous(), w, bias, 4, 4,
                                                      torch.ones(1, lens[b], device=DEV)), lens)


@pytest.mark.parametrize("L", [300, 77])
def test_masked_mean_ragged(hsv, L):
    ops = hsv.ops
    lens = [L, L - 1, 129, 128, 5, 1]
    B = len(lens)
    x = _garbage_tail(torch.randn(B, 256, L, generator=torch.Generator().manual_seed(L)).to(DEV), lens)
    out = ops.masked_mean(x, None, valid_len=_lens(lens))
    for b, n in enumerate(lens):
        assert torch.equal(out[b:b + 1], ops.masked_mean(x[b:b + 1, :, :n].contiguous(), torch.ones(1, n, device=DEV)))


def test_ln_mod_zero_masked_rows(hsv):
    ops = hsv.ops
    B, C, T = 2, 192, 131
    gen = torch.Generator().manual_seed(6)
    x = torch.randn(B, C, T, generator=gen).to(DEV)
    y = torch.randn(B, C, T, generator=gen).to(DEV)
    mod = torch.randn(B, 6 * C, generator=gen).to(DEV)
    mask = (torch.arange(T)[None, :] < torch.tensor([T, 90])[:, None]).float().to(DEV)
    a, z = ops.blk16_buffer(B, C, T, DEV, slot=8), ops.blk16_buffer(B, C, T, DEV, slot=9)
    x1, x2 = x.clone(), x.clone()
    ops.gate_ln_mod_blk16(x1, y, mod[:, :C], mod[:, C:2 * C], mod[:, 2 * C:3 * C], a, 6 * C, mask)
    ops.gate_ln_mod_blk16(x2, y, mod[:, :C], mod[:, C:2 * C], mod[:, 2 * C:3 * C], z, 6 * C, mask, zero_masked=True)
    assert torch.equal(x1, x2)
    ua, uz = ops.unpack_blk16(a, C, T), ops.unpack_blk16(z, C, T)
    assert torch.equal(uz, ua * mask.unsqueeze(1)) and bool((ua[1, :, 90:] != 0).any())


# ---------------------------------------------------------------------------------------------- modules
@pytest.fixture(scope="module")
def synthesizer(hsv):
    m = hsv.HierSpeechSynthesizer()
    m.load_state_dict(synth.synthesizer_sd(1234), strict=True)
    return m.to(DEV).eval()


LENS = [500, 437, 251, 100, 7]
PROMPTS = [150, 300, 101, 217, 64]


def _job(lens, prompts, seed=1111):
    """Per-item inputs: w2v [1,1024,n], f0 [1,1,4n], prompt pair [2,80,m] (equal-length twins), eps pair."""
    from megatts2_hierspeechpp_b200 import synthetic
    items = []
    for i, (n, m) in enumerate(zip(lens, prompts)):
        w2v, f0, mel = synthetic.synthesizer_inputs(n, m, seed=seed + i)
        items.append((w2v.to(DEV), f0.to(DEV), mel.to(DEV)))
    return items


def _batch(items, lens, prompts, T, Tm, pairs=True):
    B = len(items)
    src = torch.zeros(B, 1024, T, device=DEV)
    f0 = torch.zeros(B, 1, 4 * T, device=DEV)
    rows = 2 * B if pairs else B
    mel = torch.zeros(rows, 80, Tm, device=DEV)
    for b, ((w, f, m), n, p) in enumerate(zip(items, lens, prompts)):
        src[b, :, :n] = w[0]
        f0[b, :, :4 * n] = f[0]
        mel[b, :, :p] = m[0]
        if pairs:
            mel[B + b, :, :p] = m[1]
    tl = prompts + prompts if pairs else prompts
    return (_garbage_tail(src, lens, seed=1), _garbage_tail(f0, lens, scale=4, seed=2), _garbage_tail(mel, tl, seed=3))


def test_style_encoder_items_equal_their_own_runs(synthesizer):
    lens = [300, 299, 150, 33, 1]
    B, T = len(lens), 300
    mel = _garbage_tail(torch.randn(B, 80, T, generator=torch.Generator().manual_seed(3)).to(DEV) * 2 - 4, lens)
    with torch.no_grad():
        g = synthesizer.emb_g(mel, lengths=_lens(lens))
        for b, n in enumerate(lens):
            assert torch.equal(g[b:b + 1], synthesizer.emb_g(mel[b:b + 1, :, :n].contiguous(),
                                                             torch.ones(1, 1, n, device=DEV))), (b, n)
        assert torch.equal(synthesizer.emb_g(mel, lengths=lens), g)          # host sequence


def test_posterior_encoder_and_flows_items_equal_their_own_runs(synthesizer):
    lens = LENS
    B, T = len(lens), max(lens)
    items = _job(lens, PROMPTS)
    src, f0, _ = _batch(items, lens, PROMPTS, T, max(PROMPTS))
    g = torch.randn(B, 256, 1, generator=torch.Generator().manual_seed(8)).to(DEV)
    eps = _garbage_tail(torch.randn(B, 192, T, generator=torch.Generator().manual_seed(9)).to(DEV), lens, seed=4)
    vl = _lens(lens)
    with torch.no_grad():
        z, m, logs = synthesizer.enc_p_l(src, f0, None, g=g, eps=eps, noise_scale=0.5, lengths=vl)
        f1 = synthesizer.flow_l(z, None, g=g, reverse=True, lengths=vl)
        f2 = synthesizer.flow(f1, None, g=g, reverse=True, lengths=vl)
        # a flow passes its first half-channels' padding through (as the reference's does), but never reads it
        f1g = synthesizer.flow_l(_garbage_tail(z, lens, seed=5), None, g=g, reverse=True, lengths=vl)
        for b, n in enumerate(lens):
            one = torch.ones(1, 1, n, device=DEV)
            gb = g[b:b + 1]
            zo, mo, lo = synthesizer.enc_p_l(src[b:b + 1, :, :n].contiguous(), f0[b:b + 1, :, :4 * n].contiguous(), one,
                                             g=gb, eps=eps[b:b + 1, :, :n].contiguous(), noise_scale=0.5)
            assert torch.equal(z[b:b + 1, :, :n], zo) and bool((z[b, :, n:] == 0).all()), b
            assert torch.equal(m[b:b + 1, :, :n], mo) and torch.equal(logs[b:b + 1, :, :n], lo), b
            fo = synthesizer.flow_l(zo, one, g=gb, reverse=True)
            assert torch.equal(f1[b:b + 1, :, :n], fo) and bool((f1[b, :, n:] == 0).all()), b
            assert torch.equal(f1g[b:b + 1, :, :n], fo), b
            fo2 = synthesizer.flow(fo, one, g=gb, reverse=True)
            assert torch.equal(f2[b:b + 1, :, :n], fo2) and bool((f2[b, :, n:] == 0).all()), b


# ---------------------------------------------------------------------------------------------- whole calls
def _own_noise(seed, n, draws):
    """The draws the per_item=False method makes on one item after torch.manual_seed(seed)."""
    torch.manual_seed(seed)
    return [torch.randn(1, 192, n, device=DEV) for _ in range(draws)]


@pytest.mark.parametrize("method", ["voice_conversion_noise_control", "voice_conversion", "infer"])
def test_whole_call_items_equal_their_own_calls(synthesizer, method):
    lens, prompts = LENS, PROMPTS
    if method == "infer":
        prompts = lens                                      # x_mel shares the source's lengths
    B, T, Tm = len(lens), max(lens), max(prompts)
    items = _job(lens, prompts)
    if method == "infer":
        items = [(w, f, torch.randn(1, 80, n, generator=torch.Generator().manual_seed(n)).to(DEV) * 2 - 4)
                 for (w, f, _), n in zip(items, lens)]
    pairs = method == "voice_conversion_noise_control"
    src, f0, mel = _batch(items, lens, prompts, T, Tm, pairs=pairs)
    eps = torch.zeros(B, 192, T, device=DEV)
    for b, n in enumerate(lens):
        eps[b, :, :n] = _own_noise(100 + b, n, 1 if method == "infer" else 2)[-1][0]
    eps = _garbage_tail(eps, lens, seed=7)
    vl = _lens(lens)
    tl = _lens(prompts + prompts if pairs else prompts)
    with torch.no_grad():
        if method == "voice_conversion_noise_control":
            out = synthesizer.voice_conversion_noise_control(src, vl, mel, tl, f0, 0.333, False, 0.3, per_item=True,
                                                             eps=eps)
        elif method == "voice_conversion":
            out = synthesizer.voice_conversion(src, vl, mel, tl, f0, 0.333, per_item=True, eps=eps)
        else:
            out = synthesizer.infer(mel, src, vl, f0, per_item=True, eps=eps)[0]
        assert out.shape == (B, 1, 320 * T)

        def own(b):
            n, p = lens[b], prompts[b]
            w, f, m = items[b]
            torch.manual_seed(100 + b)
            ln = torch.LongTensor([n]).to(DEV)
            if method == "voice_conversion_noise_control":
                return synthesizer.voice_conversion_noise_control(w, ln, m, torch.LongTensor([p, p]).to(DEV), f, 0.333,
                                                                  False, 0.3)
            if method == "voice_conversion":
                return synthesizer.voice_conversion(w, ln, m[:1], torch.LongTensor([p]).to(DEV), f, 0.333)
            return synthesizer.infer(m, w, ln, f)[0]

        _check_items(out, own, lens, scale=320)


def test_batch_of_one_at_full_length_equals_the_unbatched_call(synthesizer):
    items = _job([200], [150])
    w, f, m = items[0]
    ln, ln2 = torch.LongTensor([200]).to(DEV), torch.LongTensor([150, 150]).to(DEV)
    eps = _own_noise(7, 200, 2)[-1]
    with torch.no_grad():
        got = synthesizer.voice_conversion_noise_control(w, ln, m, ln2, f, 0.333, False, 0.3, per_item=True, eps=eps)
        torch.manual_seed(7)
        ref = synthesizer.voice_conversion_noise_control(w, ln, m, ln2, f, 0.333, False, 0.3)
    assert torch.equal(got, ref)


def test_one_graph_serves_every_length_mix(hsv, synthesizer):
    B, T, Tm = 3, 120, 100
    items = _job([T] * B, [Tm] * B, seed=50)
    src, f0, mel = _batch(items, [T] * B, [Tm] * B, T, Tm)
    eps = torch.randn(B, 192, T, generator=torch.Generator().manual_seed(2)).to(DEV)

    def call(s, f, m, vl, tl, e):
        return synthesizer.voice_conversion_noise_control(s, vl, m, tl, f, 0.333, False, 0.3, per_item=True, eps=e)

    runner = hsv.CudaGraphRunner(call)
    with torch.no_grad():
        for lens, prompts in (([120, 13, 77], [100, 51, 9]), ([7, 120, 119], [99, 100, 64])):
            s, f, m = (_garbage_tail(src, lens, seed=1), _garbage_tail(f0, lens, scale=4, seed=2),
                       _garbage_tail(mel, prompts + prompts, seed=3))
            vl, tl = _lens(lens), _lens(prompts + prompts)
            got = runner(s, f, m, vl, tl, eps).clone()
            assert torch.equal(got, call(s, f, m, vl, tl, eps))
            assert all(bool((got[b, :, 320 * n:] == 0).all()) for b, n in enumerate(lens))
    assert runner.captures == 1


def test_census_per_item_variants_verified(hsv, synthesizer, monkeypatch):
    """Every conv / activation variant the per-item path launches is one tests/test_gpu_variants.py verifies."""
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

    lens, prompts = [500, 300, 120, 50], [300, 250, 200, 150]
    items = _job(lens, prompts, seed=70)
    src, f0, mel = _batch(items, lens, prompts, 500, 300)
    monkeypatch.setattr(_lib, "check", recording_check)
    with torch.no_grad():
        synthesizer.voice_conversion_noise_control(src, _lens(lens), mel, _lens(prompts + prompts), f0, 0.333, False,
                                                   0.3, per_item=True)
    torch.cuda.synchronize()
    monkeypatch.setattr(_lib, "check", orig)
    print("\n[census] per-item synthesizer: " + ", ".join(f"{k} x{n}" for k, n in sorted(seen.items())))
    assert seen
    assert not sorted(set(seen) - VERIFIED)
