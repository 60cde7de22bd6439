"""Streaming SpeechSR on the GPU: S concurrent streams through ``SpeechSRStream``, each stream's concatenated output
equal (``torch.equal``) to the offline call on the whole stream, and the stream interpolation kernel against the
full-length one at the same global indices."""
import math
import random

import numpy as np
import pytest
import torch

from conftest import golden, golden_sd
from oracle import closed_form as CF

from megatts2_hierspeechpp_b200.sr_stream import MAX_STREAM_OUTPUT

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


# ---------------------------------------------------------------------------------------------- the interpolation kernel
def _interp_window(ops, x, w, bias, o_in, W, ratio, total):
    up, down = ratio
    win = x[:, :, o_in:o_in + W].contiguous()
    vin = torch.tensor([W], dtype=torch.int32, device=DEV)
    vout = vin * up // down
    org = torch.tensor([[o_in, o_in * up // down, total]], dtype=torch.int64, device=DEV)
    return ops.sr_pre_interp_stream(win, w, bias, W * up // down, (vin, vout), org, ratio)


@pytest.mark.parametrize("ratio", [(3, 1), (3, 2)])
@pytest.mark.parametrize("where", ["start", "mid", "end", "large"])
def test_interp_stream_equals_full_length(hsv, ratio, where):
    ops = hsv.ops
    up, down = ratio
    r = up / down
    L = (MAX_STREAM_OUTPUT // up - 20) // 2 * 2 if where == "large" else 20000
    W = 4000
    o_in = {"start": 0, "mid": 9000, "end": L - W, "large": L - 3 * W}[where]
    gen = torch.Generator().manual_seed(L + o_in)
    x = torch.randn(1, 1, L, generator=gen).to(DEV)
    w = torch.randn(8, 1, 7, generator=gen).to(DEV)
    bias = torch.randn(8, generator=gen).to(DEV)
    Lout = L * up // down
    full = ops.sr_pre_interp(x, w, bias, Lout)
    at_end = o_in + W == L
    got = _interp_window(ops, x, w, bias, o_in, W, ratio, L if at_end else -1)
    edge = math.ceil(r * 5.5 + 0.5)          # every tap inside the window (stream_reach's interpolation term)
    lo = 0 if o_in == 0 else edge
    hi = W * up // down - (0 if at_end else edge)
    o_out = o_in * up // down
    assert torch.equal(got[..., lo:hi], full[..., o_out + lo:o_out + hi])
    if where == "end":
        # the clamp at the stream's total length is only applied when it is given
        unclamped = _interp_window(ops, x, w, bias, o_in, W, ratio, -1)
        assert not torch.equal(unclamped[..., hi - 2:hi], full[..., o_out + hi - 2:o_out + hi])
    # ramp probe: i0 / i1 / lambda of the global indices, as the full-length probe reads them back
    ramp = torch.arange(L, dtype=torch.float32, device=DEV).view(1, 1, L)
    delta = torch.zeros(1, 1, 7, device=DEV)
    delta[0, 0, 3] = 1.0
    probe = _interp_window(ops, ramp, delta, None, o_in, W, ratio, L if at_end else -1)[0, 0, lo:hi].double()
    i0, i1, lam = CF.linear_interp_table(L, Lout, fma=True)
    sl = slice(o_out + lo, o_out + hi)
    want = (1 - lam[sl].astype(np.float64)) * i0[sl] + lam[sl].astype(np.float64) * i1[sl]
    assert torch.equal(probe.float(), ops.sr_pre_interp(ramp, delta, None, Lout)[0, 0, o_out + lo:o_out + hi])
    torch.testing.assert_close(probe.cpu(), torch.from_numpy(want), rtol=0, atol=2e-3 * L ** 0.5)


# ---------------------------------------------------------------------------------------------- the stream module
@pytest.fixture(scope="module", params=[24, 48])
def sr(request, hsv):
    which = request.param
    m = (hsv.SpeechSR24 if which == 24 else hsv.SpeechSR48)(100, 40, **hsv.SR_CFG)
    m.load_state_dict(golden_sd(f"speechsr{which}_state.npz"), strict=True)
    return m.to(DEV).eval()


def _example():
    return torch.from_numpy(golden("speechsr24_example.npz")["x_int16"].astype(np.float32) / 32768.0)


def _run(hsv, sr, S, N, plans, seed, check=None):
    """Drive a SpeechSRStream.  ``plans[b]``: the streams slot b plays one after the other, each (audio, gap, sizes):
    ``gap`` idle steps first, then chunks of ``sizes`` (0 = an idle step of an open stream), ending on the last chunk,
    or on a flush step when sizes ends with 0.  Returns every stream's concatenated output per slot, and the stream."""
    st = hsv.SpeechSRStream(sr, S, N)
    up, down = st.ratio
    mirror = st.schedule()
    queue = [list(p) for p in plans]
    cur = [None] * S      # [audio, pos, sizes, k, outputs]
    gaps = [q[0][1] if q else 0 for q in queue]
    results = [[] for _ in range(S)]
    rng = random.Random(seed)
    steps = 0
    while any(queue) or any(c is not None for c in cur):
        x = torch.zeros(S, N)
        n_new, start, end = [0] * S, [False] * S, [False] * S
        for b in range(S):
            if cur[b] is None and queue[b]:
                if gaps[b] > 0:
                    gaps[b] -= 1
                    continue
                audio, _, sizes = queue[b].pop(0)
                cur[b] = [audio, 0, list(sizes), 0, []]
                start[b] = True
            if cur[b] is None:
                continue
            audio, pos, sizes, k, _ = cur[b]
            n = sizes[k]
            x[b, :n] = audio[pos:pos + n]
            n_new[b] = n
            cur[b][1], cur[b][3] = pos + n, k + 1
            end[b] = cur[b][3] == len(sizes)
        expect = mirror.step(n_new, start, end)
        nn = torch.tensor(n_new, dtype=torch.int32, device=DEV)
        out, n_out = st.step(x.to(DEV), nn, torch.tensor(start, device=DEV), torch.tensor(end, device=DEV, dtype=torch.int32))
        got_n = n_out.cpu().tolist()
        assert got_n == expect, (steps, got_n, expect)
        for b in range(S):
            if cur[b] is None:
                continue
            cur[b][4].append(out[b, :got_n[b]].clone())
            if not end[b]:
                # never ahead of received * ratio - lookahead
                assert sum(t.numel() for t in cur[b][4]) <= max(0, cur[b][1] * up // down - st.lookahead)
            else:
                results[b].append((cur[b][0], torch.cat(cur[b][4])))
                cur[b] = None
                gaps[b] = queue[b][0][1] if queue[b] else 0
        if check is not None:
            check(st, steps)
        steps += 1
    return results, st


def _sizes(rng, L, N, down, exact=False):
    """Random chunk sizes (some 0) summing to L, multiples of down; ``exact``: full chunks only."""
    if exact:
        return [N] * (L // N)
    out, left = [], L
    while left > 0:
        n = min(left, rng.randrange(0, N + 1, down) if rng.random() > 0.15 else 0)
        out.append(n)
        left -= n
    if rng.random() < 0.3:
        out.append(0)      # a flush step
    return out


def _check_equal(sr, results):
    n = 0
    with torch.no_grad():
        for slot in results:
            for audio, got in slot:
                ref = sr(audio.view(1, 1, -1).to(DEV))[0, 0]
                assert got.shape == ref.shape, (got.shape, ref.shape)
                assert torch.equal(got, ref), (audio.numel(), (got - ref).abs().max().item())
                n += 1
    return n


@pytest.mark.parametrize("parallel", [False, True])
@pytest.mark.parametrize("N", [160, 320, 4800])
def test_streams_equal_offline(hsv, sr, N, parallel):
    """Example audio and seeded synthetic streams in 4 slots: random n_new (including 0), different start and end
    steps, slot reuse, streams of 1-2 samples and shorter than the lookahead, one ending exactly on a chunk boundary."""
    sr.dec.parallel_blocks = parallel
    try:
        down = 2 if sr.dec.scale == 1.5 else 1
        rng = random.Random(N * 10 + parallel)
        gen = torch.Generator().manual_seed(N)

        def synth(L):
            return torch.randn(L, generator=gen) * 0.2 * torch.sin(torch.arange(L) * 0.01)

        ex = _example()
        tiny = [2] if down == 2 else [1, 2]
        plans = [
            [(ex, 0, _sizes(rng, ex.numel(), N, down))],
            [(synth(L), rng.randrange(3), _sizes(rng, L, N, down)) for L in tiny + [40, 96, 3000]],
            [(synth(4 * N), 1, _sizes(rng, 4 * N, N, down, exact=True)), (synth(30), 0, [30]),
             (synth(2 * N + 2), 2, _sizes(rng, 2 * N + 2, N, down))],
            [(synth(L), rng.randrange(4), _sizes(rng, L, N, down)) for L in (12000, 500, 64)],
        ]
        results, st = _run(hsv, sr, 4, N, plans, seed=N)
        assert _check_equal(sr, results) == 1 + len(tiny) + 3 + 3 + 3
        assert st.captures == 1
    finally:
        sr.dec.parallel_blocks = False


def test_chunk_2_on_a_short_clip(hsv, sr):
    ex = _example()[10000:10600]
    results, st = _run(hsv, sr, 2, 2, [[(ex, 0, [2] * 300)], [(ex[:100], 5, [2] * 50), (ex[:2], 0, [2])]], seed=2)
    assert _check_equal(sr, results) == 3 and st.captures == 1


def test_idle_step_changes_nothing_and_recapture(hsv, sr):
    """An all-idle step leaves the state bit for bit unchanged; after load_state_dict the next step recaptures (on an
    idle step) and the streams stay exact; invalid requests leave their slot idle."""
    N = 320
    ex = _example()
    sd = golden_sd(f"speechsr{24 if sr.dec.scale == 1.5 else 48}_state.npz")

    def check(st, step):
        if step == 20:
            S = st.slots
            hist, state = st._hist.clone(), st._state.clone()
            z = torch.zeros(S, dtype=torch.int32, device=DEV)
            out, n_out = st.step(torch.randn(S, N, device=DEV), z, z.bool(), z)
            assert not n_out.any() and not out.any()
            assert torch.equal(st._hist, hist) and torch.equal(st._state, state)
            # requests the device ignores: too many samples, an odd count at 24 kHz, an end for the closed slot 2
            bad = torch.tensor([N + 2, 3 if st.ratio[1] == 2 else N + 1, 0], dtype=torch.int32, device=DEV)
            out, n_out = st.step(torch.randn(S, N, device=DEV), bad, z.bool(),
                                 torch.tensor([0, 0, 1], dtype=torch.int32, device=DEV))
            assert not n_out.any()
            assert torch.equal(st._hist, hist) and torch.equal(st._state, state)
            assert st.captures == 1
            sr.load_state_dict(sd)
        if step == 21:
            assert st.captures == 2

    plans = [[(ex, 0, [N] * (ex.numel() // N))], [(ex[:20000], 3, [N] * (20000 // N) + [20000 % N])], []]
    results, st = _run(hsv, sr, 3, N, plans, seed=3, check=check)
    assert _check_equal(sr, results) == 2
