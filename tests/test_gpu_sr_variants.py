"""The SpeechSR-only kernels against exact and float64 references, and a census of every SpeechSR entry point.

(a) Stream bookkeeping (``hsv_sr_stream_window`` / ``hsv_sr_stream_emit``, csrc/sr_stream.cu) against a pure-Python
    int64 model written from the contract in include/hsv.h (not from ``sr_stream.SRStreamSchedule``).  Seeded random
    traffic drives the two kernels directly, with a synthetic ``y`` in place of the SpeechSR forward; after every step
    ``win``, the valid lengths, ``origin``, ``plan``, ``out``, ``n_out``, ``hist`` and ``state`` must equal the model bit
    for bit.  ``x_new`` past ``n_new`` and ``y`` outside the emit range are NaN, and the part of ``hist`` no stream has
    filled holds a NaN sentinel: reading any of them, or overwriting the sentinel, changes a compared bit.  A CPU test
    shows that the traffic reaches every kind of request and that three defective models are told apart from the
    model.
(b) ``hsv_sr_pre_interp_stream`` with many slots in one launch against float64: per slot its own stream, origin
    (0, small, mid-stream, near ``MAX_STREAM_OUTPUT``), valid length (0, 1, 2, < 7, the window) and total length (-1
    or the stream's).  The reference is conv_pre in float64 on the stream with the taps outside the window zeroed,
    interpolated at the global indices with the kernel's fp32 table; the bound is derived in ``_interp_ref``.  Every
    output whose taps all lie inside the window must also equal the full-length ``sr_pre_interp`` bit for bit.  A CPU
    emulation shows that a window-relative lambda and a missing last-window clamp fail the bound.
(c) ``peak_norm_pcm16`` / ``peak_norm_pcm16_rows`` bit for bit against the reference's fp32 expression
    (``OF.peak_norm_pcm16``) at the edges: one prompt peak per row, the global-peak fold over 1, 33 and 300 rows, a
    row longer than the 148 x 8-CTA grid covers in one pass, peaks at either end, negative peaks, +-0, rows zero past
    a ragged length, and inputs built so that the scaled value lies within an fp32 ulp of an integer (a CPU test shows
    that a reciprocal multiply, a pre-folded s1 * s2, an unrounded s1 product and round-to-nearest each change the
    int16 output there).  All-zero rows give 0 (documented in ``ops.peak_norm_pcm16``).
(d) The ragged activation is checked in test_gpu_variants.py (``act:R{R}:{mode}:ragged``).
(e) Census: the conv, activation, CUDA-core conv, attention and frame-op launches of the SpeechSR24 / SpeechSR48 /
    chain24 benchmark workloads, a ragged SpeechSR24 batch, ``SpeechSRStream`` at both rates, and (conv / activation)
    the ragged vocoder / SpeechSR48 / text-to-vec batches and a per-item synthesizer batch must all be keys the four
    variant files verify.
"""
import argparse
import functools
import os
import random
import sys

import numpy as np
import pytest
import torch

from oracle import functional as OF

DEV = "cuda:0"
U32 = 2.0 ** -24
RATIOS = ((3, 1), (3, 2))


def _bits(t):
    """The raw bits of a float32 tensor (NaN payloads included) as a numpy int32 array."""
    return t.detach().cpu().contiguous().view(torch.int32).numpy()


def _f32(a):
    return np.asarray(a, np.float32)


# ----------------------------------------------------------------------------------------------
# (a) stream bookkeeping: the model
# ----------------------------------------------------------------------------------------------
HIST_SENTINEL = np.int32(0x7FC5A5A5)      # a quiet NaN with a payload: hist entries no stream has written yet


@functools.lru_cache(maxsize=None)
def shipped(ratio):
    """(history H, lookahead) of the SpeechSR generator of this ratio, as SpeechSRStream derives them."""
    from megatts2_hierspeechpp_b200 import SR_CFG, SpeechSR24, SpeechSR48
    from megatts2_hierspeechpp_b200.sr_stream import history_len, stream_reach
    gen = (SpeechSR48 if ratio == (3, 1) else SpeechSR24)(100, 40, **SR_CFG).dec
    la, halo = stream_reach(gen)
    return history_len(la, halo, ratio), la


class StreamModel:
    """include/hsv.h's hsv_sr_stream_window / hsv_sr_stream_emit in Python integers.

    Per slot: received, emitted, open.  A request is ignored (n = 0, no flags) when n < 0, n > N, n % down != 0, or it
    carries samples or an end for a closed slot without start.  ``defect`` selects a deliberately wrong variant for the
    CPU test that shows the traffic tells them apart."""

    def __init__(self, S, N, H, ratio, lookahead, defect=None):
        self.S, self.N, self.H, self.la, self.defect = S, N, H, lookahead, defect
        self.up, self.down = ratio
        self.recv, self.emitted, self.open = [0] * S, [0] * S, [0] * S
        self.hist = np.full((S, H), HIST_SENTINEL, np.int32)           # bits
        self.kinds = {}

    def _count(self, k):
        self.kinds[k] = self.kinds.get(k, 0) + 1

    def _classify(self, b, n, s, e):
        op = self.open[b]
        if n == 0 and not s and not e:
            self._count("n = 0 chunk on open stream" if op else "idle")
        elif n < 0:
            self._count("invalid n < 0")
        elif n > self.N:
            self._count("invalid n > N")
        elif n % self.down:
            self._count("invalid n % down")
        elif not op and not s:
            self._count("invalid end on closed slot" if e and n == 0 else "invalid samples on closed slot")
        else:
            if s and op:
                self._count("start on open slot")
            if s and e and n == 0:
                self._count("start + end with n = 0")
            if op and not s and n == 0 and e:
                self._count("flush (end with n = 0)")
            if s and self.recv[b] == 0 and not op and self.kinds.get(f"closed{b}"):
                self._count("slot reuse")

    def _plan(self, b, n, s, e):
        H, up, down = self.H, self.up, self.down
        op = bool(self.open[b])
        invalid = n < 0 or n > self.N or n % down != 0 or (not op and not s and (n > 0 or e))
        if self.defect == "invalid end applied":
            invalid = n < 0 or n > self.N or n % down != 0 or (not op and not s and n > 0)
        if invalid:
            n, s, e = 0, False, False
        keep = s and self.defect == "start keeps history"
        recv0 = self.recv[b] if (not s or keep) else 0
        emit0 = self.emitted[b] if (not s or keep) else 0
        hlen = min(recv0, H)
        o_in = recv0 - hlen
        recv1 = recv0 + n
        live = op or s
        full = recv1 * up // down
        if not live:
            emit1 = emit0
        elif e:
            emit1 = full
        else:
            emit1 = max(full - self.la, emit0)
        return dict(n=n, hlen=hlen, o_in=o_in, o_out=o_in * up // down, total=recv1 if e else -1, emit0=emit0,
                    emit1=emit1, recv1=recv1, wlen=hlen + n, open1=int(live and not e), update=int(s or e or n > 0))

    def window(self, x_bits, n_new, start, end):
        """x_bits: int32 [S, N] (bits of x_new).  Returns the expected (win bits, vin, vout, origin, plan)."""
        S, N, H = self.S, self.N, self.H
        W = H + N
        win = np.zeros((S, W), np.int32)
        vin, vout = np.zeros(S, np.int32), np.zeros(S, np.int32)
        origin, plan = np.zeros((S, 3), np.int64), np.zeros((S, 6), np.int64)
        self.plans = []
        for b in range(S):
            self._classify(b, n_new[b], start[b], end[b])
            p = self._plan(b, n_new[b], bool(start[b]), bool(end[b]))
            self.plans.append(p)
            win[b, :p["hlen"]] = self.hist[b, H - p["hlen"]:]
            win[b, p["hlen"]:p["wlen"]] = x_bits[b, :p["n"]]
            wl = p["wlen"] if p["emit1"] > p["emit0"] else 0
            vin[b], vout[b] = wl, wl * self.up // self.down
            origin[b] = (p["o_in"], p["o_out"], p["total"])
            plan[b] = (p["emit0"], p["emit1"], p["recv1"], p["wlen"], p["open1"], p["update"])
        self.win = win
        return win, vin, vout, origin, plan

    def emit_range(self, b):
        """(first window-relative output, count) the emit step copies for slot b."""
        p = self.plans[b]
        return p["emit0"] - p["o_out"], p["emit1"] - p["emit0"]

    def emit(self, y_bits, cap):
        S, H = self.S, self.H
        out = np.zeros((S, cap), np.int32)
        n_out = np.zeros(S, np.int32)
        for b, p in enumerate(self.plans):
            first, ne = self.emit_range(b)
            out[b, :ne] = y_bits[b, first:first + ne]
            n_out[b] = ne
            if p["update"]:
                if p["open1"]:
                    h1 = min(p["recv1"], H)
                    lo = 0 if self.defect == "history from the window start" else p["wlen"] - h1
                    self.hist[b, H - h1:] = self.win[b, lo:lo + h1]
                    self.recv[b], self.emitted[b], self.open[b] = p["recv1"], p["emit1"], 1
                else:
                    self.recv[b], self.emitted[b], self.open[b] = 0, 0, 0
                    self.kinds[f"closed{b}"] = 1
        return out, n_out

    def state(self):
        return np.array([self.recv, self.emitted, self.open], np.int64).T.copy()


def traffic(rng, model):
    """One step's (n_new, start, end) for every slot: idle slots, valid chunks (n = 0 included), starts on open and
    closed slots, ends and flushes, and every kind of invalid request.  Streams live long enough to fill the history
    (about 4 H / N steps)."""
    S, N, down = model.S, model.N, model.down
    life = max(1.0, 4.0 * model.H / N)
    p_end, p_restart = min(0.03, 0.6 / life), min(0.04, 0.4 / life)
    n_new, start, end = [0] * S, [0] * S, [0] * S
    if rng.random() < 0.05:
        return n_new, start, end                         # an all-idle step
    for b in range(S):
        if rng.random() < 0.15:
            continue                                     # an idle slot
        r = rng.random()
        if not model.open[b]:
            if r < 0.5:                                  # a new stream (its first chunk may be empty)
                start[b], n_new[b], end[b] = 1, rng.randrange(0, N + 1, down), int(rng.random() < 0.05)
            elif r < 0.6:
                start[b], end[b] = 1, 1                  # start + end with n = 0
            elif r < 0.75:
                n_new[b] = rng.randrange(down, N + 1, down)      # samples for a closed slot
            elif r < 0.9:
                end[b] = 1                               # an end for a closed slot
            else:
                start[b], n_new[b] = 1, N + down         # a start with too many samples
            continue
        start[b] = int(rng.random() < p_restart)
        end[b] = int(rng.random() < p_end)
        if r < 0.65:
            n_new[b] = rng.randrange(down, N + 1, down)
        elif r < 0.8:
            n_new[b] = 0
        elif r < 0.86:
            n_new[b] = N + rng.choice((1, down, 100))
        elif r < 0.9:
            n_new[b] = -rng.choice((1, down))
        elif r < 0.95 and down > 1:
            n_new[b] = rng.randrange(1, N, 2)
        else:
            n_new[b] = N
    return n_new, start, end


# (ratio, H, N): the shipped history with W = H + N > 256 and cap > H, the shipped history with cap < H, and a longer
# history (H > 256, cap < H) so that the emit launch's history span runs over several CTAs
def _bookkeeping_cases():
    cases = []
    for ratio in RATIOS:
        H, _ = shipped(ratio)
        cases.append((ratio, H, 320))
        cases.append((ratio, 600, 40))
    cases.append(((3, 2), shipped((3, 2))[0], 8))
    return cases


STREAM_STEPS = 500
STREAM_SLOTS = 7


def test_bookkeeping_cases_cover_both_spans():
    """The cases put W > 256 with cap > H, cap < H with the shipped history, and a history span over several CTAs."""
    seen = set()
    for ratio, H, N in _bookkeeping_cases():
        up, down = ratio
        cap = shipped(ratio)[1] + -(-N * up // down)
        seen.add(("W>256,cap>H" if H + N > 256 and cap > H else None))
        seen.add(("cap<H shipped" if cap < H and H == shipped(ratio)[0] else None))
        seen.add(("hist span > 1 CTA" if cap < H and H > 256 else None))
    assert seen - {None} == {"W>256,cap>H", "cap<H shipped", "hist span > 1 CTA"}


def _run_model(ratio, H, N, seed, defect=None):
    la = shipped(ratio)[1]
    m = StreamModel(STREAM_SLOTS, N, H, ratio, la, defect)
    rng = random.Random(seed)
    x_rng = np.random.default_rng(seed)
    up, down = ratio
    Lout = (H + N) * up // down
    cap = la + -(-N * up // down)
    trace = []
    for _ in range(STREAM_STEPS):
        n_new, start, end = traffic(rng, m)
        x = _stream_x(x_rng, n_new, STREAM_SLOTS, N)
        exp = m.window(x.view(np.int32), n_new, start, end)
        y = _stream_y(x_rng, m, Lout)
        out = m.emit(y.view(np.int32), cap)
        trace.append((exp, out, m.hist.copy(), m.state()))
    return m, trace


def _stream_x(x_rng, n_new, S, N):
    x = x_rng.standard_normal((S, N)).astype(np.float32)
    for b, n in enumerate(n_new):
        x[b, max(n, 0):] = np.nan                     # past n_new: never read
    return x


def _stream_y(x_rng, m, Lout):
    y = np.full((m.S, Lout), np.nan, np.float32)       # outside each slot's emit range: never read
    for b in range(m.S):
        first, ne = m.emit_range(b)
        y[b, first:first + ne] = x_rng.standard_normal(ne).astype(np.float32)
    return y


@pytest.mark.parametrize("ratio", RATIOS, ids=["48k", "24k"])
def test_traffic_covers_every_request_kind(ratio):
    H, _ = shipped(ratio)
    kinds = set()
    for i, (r, H, N) in enumerate(_bookkeeping_cases()):
        if r == ratio:
            m, _ = _run_model(r, H, N, seed=i)
            kinds |= {k for k in m.kinds if not k.startswith("closed")}
    want = {"idle", "invalid n < 0", "invalid n > N", "invalid end on closed slot", "invalid samples on closed slot",
            "start on open slot", "start + end with n = 0", "n = 0 chunk on open stream", "flush (end with n = 0)",
            "slot reuse"}
    if ratio[1] == 2:
        want.add("invalid n % down")
    assert want <= kinds, sorted(want - kinds)


@pytest.mark.parametrize("defect", ["start keeps history", "invalid end applied", "history from the window start"])
def test_model_tells_defects_apart(defect):
    """A model with a plausible defect differs from the model, on the same traffic, in some compared output."""
    ratio, H, N = _bookkeeping_cases()[0]
    _, good = _run_model(ratio, H, N, seed=0)
    _, bad = _run_model(ratio, H, N, seed=0, defect=defect)

    def same(a, b):
        if isinstance(a, tuple):
            return all(same(u, v) for u, v in zip(a, b))
        return np.array_equal(a, b)

    assert not all(same(g, b) for g, b in zip(good, bad))


@pytest.mark.gpu
@pytest.mark.parametrize("ratio,H,N", _bookkeeping_cases(), ids=lambda v: str(v).replace(" ", ""))
def test_stream_bookkeeping_vs_model(hsv, ratio, H, N):
    ops = hsv.ops
    la = shipped(ratio)[1]
    S = STREAM_SLOTS
    seed = H * 7 + N + ratio[1]
    m = StreamModel(S, N, H, ratio, la)
    rng = random.Random(seed)
    x_rng = np.random.default_rng(seed)
    up, down = ratio
    W, cap = H + N, la + -(-N * up // down)
    Lout = W * up // down
    hist = torch.from_numpy(m.hist.copy()).view(torch.float32).to(DEV)
    state = torch.zeros(S, 3, dtype=torch.int64, device=DEV)

    def i32(v):
        return torch.tensor(v, dtype=torch.int32, device=DEV)

    for step in range(STREAM_STEPS):
        n_new, start, end = traffic(rng, m)
        x = _stream_x(x_rng, n_new, S, N)
        want = m.window(x.view(np.int32), n_new, start, end)
        got = ops.sr_stream_window(torch.from_numpy(x).to(DEV), i32(n_new), i32(start), i32(end), hist, state, ratio,
                                   la)
        for name, g, w in zip(("win", "vin", "vout", "origin", "plan"), got, want):
            g = _bits(g) if g.dtype == torch.float32 else g.cpu().numpy()
            assert np.array_equal(g, w), (step, name, np.argwhere(g != w)[:4].tolist(), n_new, start, end)
        y = _stream_y(x_rng, m, Lout)
        out, n_out = ops.sr_stream_emit(torch.from_numpy(y).to(DEV), got[0], got[3], got[4], hist, state, cap)
        w_out, w_n = m.emit(y.view(np.int32), cap)
        assert np.array_equal(n_out.cpu().numpy(), w_n), (step, n_out.cpu().tolist(), w_n.tolist())
        assert np.array_equal(_bits(out), w_out), (step, "out")
        assert np.array_equal(_bits(hist), m.hist), (step, "hist", np.argwhere(_bits(hist) != m.hist)[:4].tolist())
        assert np.array_equal(state.cpu().numpy(), m.state()), (step, state.cpu().tolist(), m.state().tolist())
    # the traffic opened streams long enough to fill the history and reached the idle paths
    assert m.kinds.get("idle", 0) > 0 and (m.hist != HIST_SENTINEL).all(axis=1).any()


# ----------------------------------------------------------------------------------------------
# (b) sr_pre_interp_stream, many slots in one launch
# ----------------------------------------------------------------------------------------------
def _interp_at(g, scale, L_clamp):
    """i0, i1, lambda of CF.linear_interp_table(fma=True) at output indices g (int64 array), with the stream's fp32
    scale and the Lin - 1 clamp at L_clamp (None: no clamp, a stream whose length is not yet known)."""
    dst = g.astype(np.float32) + np.float32(0.5)
    src = (np.float64(scale) * dst.astype(np.float64) - 0.5).astype(np.float32)     # one rounding: the FMA
    src = np.maximum(src, np.float32(0.0))
    i0 = src.astype(np.int64)
    if L_clamp is not None:
        i0 = np.minimum(i0, L_clamp - 1)
        i1 = i0 + (i0 < L_clamp - 1)
    else:
        i1 = i0 + 1
    return i0, i1, (src - i0.astype(np.float32)).astype(np.float32)


def test_interp_at_equals_the_oracle_table():
    from oracle import closed_form as CF
    for L, Lout in ((600, 1800), (600, 900), (7, 21), (2, 3)):
        want = CF.linear_interp_table(L, Lout, fma=True)
        got = _interp_at(np.arange(Lout), np.float32(np.float32(L) / np.float32(Lout)), L)
        for a, b in zip(got, want):
            assert np.array_equal(a, b)


def _taps(xs, lo, o_in, vin, L):
    """x of the stream at indices lo[:, None] + 0..6, zero outside the window [o_in, o_in + vin) and the stream."""
    idx = lo[:, None] + np.arange(7)[None, :]
    ok = (idx >= o_in) & (idx < o_in + vin) & (idx >= 0) & (idx < L)
    return np.where(ok, xs(np.clip(idx, 0, L - 1)), 0.0)


def _interp_ref(xs, L, o_in, vin, total, w, bias, up, down):
    """float64 reference and bound of one window's outputs [C, vout]: conv_pre of the window's taps (zero outside it),
    interpolated at the global indices o_out + t with the fp32 table.

    Bound: each 7-tap sum is 7 fmaf roundings plus the bias add, <= 8 u S (S = sum |w x| + |b|); 1 - lambda rounds
    once (<= u |va|); the blend w0 va + w1 vb rounds at most twice (<= 2 u ((1 - l) S_a + l S_b)).  Together
    <= u (10 ((1 - l) S_a + l S_b) + S_a), with 1 % slack for the second-order terms."""
    vout = vin * up // down
    g = o_in * up // down + np.arange(vout, dtype=np.int64)
    scale = np.float32(down) / np.float32(up)
    i0, i1, lam = _interp_at(g, scale, total if total >= 0 else None)
    xa = _taps(xs, i0 - 3, o_in, vin, L)
    xb = _taps(xs, i1 - 3, o_in, vin, L)
    w64, b64 = w.astype(np.float64), bias.astype(np.float64)
    va = xa @ w64.T + b64                         # [vout, C]
    vb = xb @ w64.T + b64
    sa = np.abs(xa) @ np.abs(w64).T + np.abs(b64)
    sb = np.abs(xb) @ np.abs(w64).T + np.abs(b64)
    l64 = lam.astype(np.float64)[:, None]
    ref = (1 - l64) * va + l64 * vb
    bound = 1.01 * U32 * (10 * ((1 - l64) * sa + l64 * sb) + sa) + 1e-30
    inside = ((i0 - 3 >= o_in) | (o_in == 0)) & ((i1 + 3 < o_in + vin) | ((o_in + vin == L) & (total == L)))
    return ref.T, bound.T, inside, (i0, i1, lam)


def _emulate_window(xs, L, o_in, vin, total, w, bias, up, down, lam_mode="global", clamp=True):
    """fp32 emulation of the stream kernel's arithmetic (fmaf chains, 1 - lambda, the blend), optionally with a
    window-relative lambda or without the last-window clamp."""
    vout = vin * up // down
    t = np.arange(vout, dtype=np.int64)
    scale = np.float32(down) / np.float32(up)
    if lam_mode == "global":
        i0, i1, lam = _interp_at(o_in * up // down + t, scale, total if (total >= 0 and clamp) else None)
    else:
        i0, i1, lam = _interp_at(t, scale, None)
        i0, i1 = i0 + o_in, i1 + o_in
    xa = _taps(xs, i0 - 3, o_in, vin, L).astype(np.float32)
    xb = _taps(xs, i1 - 3, o_in, vin, L).astype(np.float32)
    out = np.zeros((w.shape[0], vout), np.float32)
    for c in range(w.shape[0]):
        va = np.zeros(vout, np.float32)
        vb = np.zeros(vout, np.float32)
        for j in range(7):
            va = (w[c, j].astype(np.float64) * xa[:, j] + va).astype(np.float32)
            vb = (w[c, j].astype(np.float64) * xb[:, j] + vb).astype(np.float32)
        va, vb = va + bias[c], vb + bias[c]
        w0 = np.float32(1) - lam
        out[c] = (w0.astype(np.float64) * va + (lam * vb).astype(np.float64)).astype(np.float32)
    return out


MAX_OUT = 1 << 24


def _streams(down):
    """Stream lengths (multiples of down, up * L < 2^24) and the slots' windows (stream, o_in, vin, total)."""
    up = 3
    big = (MAX_OUT // up - 40) // down * down
    lens = {"A": 600, "B": 20000, "C": big, "D": 300}
    W = 400
    slots = [("A", 0, W, -1), ("A", 0, 0, -1), ("A", 0, 1, -1), ("A", 2 * down, 2, -1), ("A", 5 * down, 6, -1),
             ("A", 400, 200, 600), ("A", 400, 200, -1), ("B", 9000, W, -1), ("B", 20000 - W, W, 20000),
             ("C", big - W, W, big), ("C", big - 3 * W, W, -1), ("C", big - 2, 2, big), ("D", 0, 300, 300),
             ("B", 30 * down, 5, -1)]
    return lens, slots, W


def _stream_data(name, L, seed):
    """Deterministic stream samples by index (the long stream is never materialised on the host)."""
    def xs(idx):
        rng = np.random.default_rng(seed)
        base = rng.standard_normal(4096).astype(np.float32) * 0.5
        return base[(idx * 2654435761) % 4096].astype(np.float64) * (1 + (idx % 7) * 0.125)
    return xs


def _weights(C, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((C, 7)).astype(np.float32) * 0.4, rng.standard_normal(C).astype(np.float32) * 0.1


@pytest.mark.parametrize("down", [1, 2])
def test_interp_bound_rejects_relative_lambda_and_missing_clamp(down):
    """The fp32 emulation of the kernel meets the bound on every slot; a window-relative lambda fails it on the
    mid-stream and near-2^24 windows, and dropping the last-window clamp fails it on the windows that end a stream."""
    up = 3
    lens, slots, _ = _streams(down)
    w, bias = _weights(4, down)
    fails = {"relative": set(), "no clamp": set()}
    for k, (name, o_in, vin, total) in enumerate(slots):
        L = lens[name]
        xs = _stream_data(name, L, ord(name))
        ref, bound, _, _ = _interp_ref(xs, L, o_in, vin, total, w, bias, up, down)
        ok = _emulate_window(xs, L, o_in, vin, total, w, bias, up, down)
        assert (np.abs(ok - ref) <= bound).all(), (k, np.abs(ok - ref).max())
        for mut, kw in (("relative", dict(lam_mode="relative")), ("no clamp", dict(clamp=False))):
            bad = _emulate_window(xs, L, o_in, vin, total, w, bias, up, down, **kw)
            if (np.abs(bad - ref) > bound).any():
                fails[mut].add(k)
    mid_and_big = {k for k, s in enumerate(slots) if s[0] in "BC" and s[2] == 400}
    assert mid_and_big <= fails["relative"], (mid_and_big, fails["relative"])
    ends = {k for k, s in enumerate(slots) if s[3] >= 0}
    assert ends <= fails["no clamp"], (ends, fails["no clamp"])


@pytest.mark.gpu
@pytest.mark.parametrize("down", [1, 2], ids=["48k", "24k"])
def test_sr_pre_interp_stream_many_slots_vs_fp64(hsv, down):
    ops = hsv.ops
    up = 3
    lens, slots, W = _streams(down)
    C = 4
    w, bias = _weights(C, 10 + down)
    B = len(slots)
    x = np.full((B, 1, W), np.nan, np.float32)               # past valid_len_in: never read
    for b, (name, o_in, vin, total) in enumerate(slots):
        xs = _stream_data(name, lens[name], ord(name))
        x[b, 0, :vin] = xs(np.arange(o_in, o_in + vin)).astype(np.float32)
    vin = torch.tensor([s[2] for s in slots], dtype=torch.int32, device=DEV)
    vout = vin * up // down
    org = torch.tensor([[o, o * up // down, t] for _, o, _, t in slots], dtype=torch.int64, device=DEV)
    wt, bt = torch.from_numpy(w).view(C, 1, 7).to(DEV), torch.from_numpy(bias).to(DEV)
    Lout = W * up // down
    got = ops.sr_pre_interp_stream(torch.from_numpy(x).to(DEV), wt, bt, Lout, (vin, vout), org, (up, down)).cpu()
    full = {}
    for name, L in lens.items():
        xs = _stream_data(name, L, ord(name))
        if name == "C":      # only the tail of the long stream is used: zeros before it change no compared output
            head = L - 3 * W - 64
            xa = np.zeros(L, np.float32)
            xa[head:] = xs(np.arange(head, L)).astype(np.float32)
        else:
            xa = xs(np.arange(L)).astype(np.float32)
        full[name] = ops.sr_pre_interp(torch.from_numpy(xa).view(1, 1, L).to(DEV), wt, bt, L * up // down)
    n_inside = 0
    for b, (name, o_in, vi, total) in enumerate(slots):
        L = lens[name]
        vo = vi * up // down
        assert bool((got[b, :, vo:] == 0).all()), (b, "nonzero past valid_len_out")
        if vo == 0:
            continue
        ref, bound, inside, _ = _interp_ref(_stream_data(name, L, ord(name)), L, o_in, vi, total, w, bias, up, down)
        err = np.abs(got[b, :, :vo].double().numpy() - ref)
        assert (err <= bound).all(), (b, slots[b], err.max(), np.argwhere(err > bound)[:4].tolist())
        o_out = o_in * up // down
        idx = torch.from_numpy(np.nonzero(inside)[0])
        want = full[name][0, :, o_out:o_out + vo].cpu()[:, idx]
        assert torch.equal(got[b][:, idx], want), (b, slots[b])
        n_inside += idx.numel()
    assert n_inside > 0


# ----------------------------------------------------------------------------------------------
# (c) int16 PCM
# ----------------------------------------------------------------------------------------------
S1 = np.float32(32767.0)


def _pcm_variants(x, p, s2):
    """int16 of ((x / p) * s1) * s2 and of four plausible defects, in fp32 as numpy rounds it (IEEE, per operation)."""
    x, p, s2 = _f32(x), np.float32(p), np.float32(s2)
    q = x / p
    ok = (q * S1) * s2
    sat = lambda v: np.clip(np.trunc(np.nan_to_num(v)), -32768, 32767).astype(np.int16)
    return {
        "kernel": sat(ok),
        "reciprocal multiply": sat((x * (np.float32(1) / p)) * S1 * s2),
        "pre-folded s1 * s2": sat(q * (S1 * s2)),
        "unrounded q * s1": sat((q.astype(np.float64) * np.float64(S1) * np.float64(s2)).astype(np.float32)),
        "round to nearest": np.clip(np.rint(ok), -32768, 32767).astype(np.int16),
    }


def _near_integer_row(p, s2, L, seed):
    """A row with peak p (at index 0) whose other samples put ((x / p) * s1) * s2 within an fp32 ulp or two of an
    integer, chosen so that each defect of _pcm_variants changes at least a few of them."""
    rng = np.random.default_rng(seed)
    p, s2 = np.float32(p), np.float32(s2)
    k = rng.integers(-32000, 32000, 20000).astype(np.float64)
    x0 = _f32(k * np.float64(p) / (np.float64(S1) * np.float64(s2)))
    cand = np.concatenate([x0 + np.float32(d) * np.spacing(np.abs(x0)) for d in range(-3, 4)]).astype(np.float32)
    cand = cand[np.abs(cand) < p]
    v = _pcm_variants(cand, p, s2)
    ok = (cand / p * S1) * s2
    near = np.abs(ok - np.rint(ok)) <= 2 * np.spacing(np.abs(ok).astype(np.float32))
    pick = []
    for name, q in v.items():
        if name != "kernel":
            sel = np.nonzero((q != v["kernel"]) & near)[0]
            pick.append(cand[sel[: (L - 1) // 4]])
    body = np.concatenate(pick)
    row = np.zeros(L, np.float32)
    row[0] = p
    row[1:1 + body.size] = body[: L - 1]
    return row


PCM_S2 = (0.999, 0.5371, 0.8130001, 0.7777)


def _pcm_rows(L=4096):
    rows = [_near_integer_row(0.7318 + 0.05 * i, s2, L, i) for i, s2 in enumerate(PCM_S2)]
    return np.stack(rows), np.array(PCM_S2, np.float32)


def test_pcm_rows_catch_every_defect():
    """On the near-integer rows each defect changes the int16 output, and the numpy fp32 expression equals the
    reference's (OF.peak_norm_pcm16) bit for bit."""
    x, s2 = _pcm_rows()
    for r in range(x.shape[0]):
        v = _pcm_variants(x[r], x[r, 0], s2[r])
        ref = OF.peak_norm_pcm16(torch.from_numpy(x[r]), 32767.0, float(s2[r]))
        assert np.array_equal(v["kernel"], ref)
        for name, q in v.items():
            if name != "kernel":
                assert (q != v["kernel"]).sum() >= 3, (r, name)


def _edge_rows(L, seed):
    """Rows with the peak at the first / last sample, a negative peak, +-0 and rows zero past a ragged length."""
    rng = np.random.default_rng(seed)
    x = (np.tanh(rng.standard_normal((6, L))) * 0.6).astype(np.float32)
    x[0, 0] = 0.93
    x[1, -1] = -0.97                   # negative peak at the last sample
    x[2, L // 3] = -0.9999
    x[3, ::5] = 0.0
    x[3, 1::5] = -0.0
    x[3, 7] = 0.5
    x[4, L // 2:] = 0.0                # zero past a ragged length
    x[5, 1:] = -0.0
    x[5, 0] = -0.25
    return x


def _ref_rows(x, s2):
    return np.stack([OF.peak_norm_pcm16(torch.from_numpy(x[r]), 32767.0, float(s2[r])) for r in range(x.shape[0])])


@pytest.mark.gpu
def test_pcm16_rows_vs_reference(hsv):
    ops = hsv.ops
    xn, s2n = _pcm_rows()
    xe = _edge_rows(xn.shape[1], 5)
    x = np.concatenate([xn, xe])
    s2 = np.concatenate([s2n, np.linspace(0.3, 1.0, xe.shape[0]).astype(np.float32)])
    pcm, peaks = ops.peak_norm_pcm16_rows(torch.from_numpy(x).to(DEV), torch.from_numpy(s2).to(DEV))
    assert np.array_equal(pcm.cpu().numpy(), _ref_rows(x, s2))
    assert np.array_equal(peaks.cpu().numpy(), np.abs(x).max(axis=1))
    # the scalar-s2 per-row kernel on the same rows, row by row
    for r in range(x.shape[0]):
        one, _ = ops.peak_norm_pcm16(torch.from_numpy(x[r:r + 1]).to(DEV), 32767.0, float(s2[r]), per_row=True)
        assert torch.equal(one[0], pcm[r])


@pytest.mark.gpu
@pytest.mark.parametrize("rows", [1, 33, 300])
def test_pcm16_global_peak_fold_vs_reference(hsv, rows):
    """per_row=False: one peak over every row (rowmax_kernel's 32-thread loop over the row peaks); the largest |x|
    sits in the last row, a negative one in row 32 must lose to it."""
    ops = hsv.ops
    L = 1031
    rng = np.random.default_rng(rows)
    x = (np.tanh(rng.standard_normal((rows, L))) * 0.5).astype(np.float32)
    x[-1, L - 1] = -0.871
    if rows > 32:
        x[32, 3] = 0.8709999
    xt = torch.from_numpy(x)
    pcm, peak = ops.peak_norm_pcm16(xt.to(DEV), 32767.0, 0.999)
    assert float(peak[0]) == np.float32(0.871)
    want = OF.peak_norm_pcm16(xt, 32767.0, 0.999).reshape(rows, L)
    assert np.array_equal(pcm.cpu().numpy(), want)


@pytest.mark.gpu
def test_pcm16_long_row_grid_stride(hsv):
    """Rows longer than 148 x 8 CTAs x 2048 samples: the capped grid's loops run past their first pass, for the peak
    and the quantisation, in both the per-row and the per-row-s2 launches."""
    ops = hsv.ops
    L = 148 * 8 * 2048 + 777
    rng = np.random.default_rng(1)
    x = (rng.standard_normal((2, L)) * 0.2).astype(np.float32)
    x[0, L - 1] = 1.7                  # the peak in the last grid-stride pass
    x[1, L - 2049] = -1.9
    s2 = np.array([0.999, 0.61], np.float32)
    xt = torch.from_numpy(x).to(DEV)
    pcm, peaks = ops.peak_norm_pcm16_rows(xt, torch.from_numpy(s2).to(DEV))
    assert np.array_equal(peaks.cpu().numpy(), np.float32([1.7, 1.9]))
    assert np.array_equal(pcm.cpu().numpy(), _ref_rows(x, s2))
    pr, _ = ops.peak_norm_pcm16(xt, 32767.0, 0.999, per_row=True)
    assert torch.equal(pr[0], pcm[0])


@pytest.mark.gpu
def test_pcm16_all_zero_rows_give_zero(hsv):
    """An all-zero row has peak 0: 0 / 0 is NaN, which the device's float-to-int conversion makes 0 (the docstring of
    ops.peak_norm_pcm16).  Not compared with numpy, whose NaN -> int16 cast is platform-defined; the other rows of a
    per-row batch are unaffected."""
    ops = hsv.ops
    x = _edge_rows(777, 9)
    x[2] = 0.0
    x[4, :] = -0.0
    s2 = np.linspace(0.5, 1.0, x.shape[0]).astype(np.float32)
    pcm, peaks = ops.peak_norm_pcm16_rows(torch.from_numpy(x).to(DEV), torch.from_numpy(s2).to(DEV))
    pcm = pcm.cpu().numpy()
    assert not pcm[2].any() and not pcm[4].any()
    assert float(peaks[2]) == 0.0 and float(peaks[4]) == 0.0
    keep = [0, 1, 3, 5]
    assert np.array_equal(pcm[keep], _ref_rows(x[keep], s2[keep]))
    z, _ = ops.peak_norm_pcm16(torch.zeros(3, 100, device=DEV), 32767.0, 0.999)
    assert not z.any()


# ----------------------------------------------------------------------------------------------
# (e) census
# ----------------------------------------------------------------------------------------------
def _families(ops):
    """{family: (calls, key function, verified set)} from the four variant files."""
    from test_gpu_direct_variants import _DIRECT_CALLS, VERIFIED as DIRECT_VERIFIED, direct_key
    from test_gpu_front_variants import _MHA_CALLS, FRONT_VERIFIED, mha_key
    from test_gpu_variants import _CONV_CALLS, VERIFIED, act_key, conv_key
    return {
        ops.LAUNCH_CONV: (set(_CONV_CALLS) | {"hsv_conv1d_umma_astride"}, conv_key, VERIFIED),
        ops.LAUNCH_ACT: ({"hsv_act1d_snakebeta"}, act_key, VERIFIED),
        ops.LAUNCH_DIRECT: (set(_DIRECT_CALLS), direct_key, DIRECT_VERIFIED),
        ops.LAUNCH_MHA: (set(_MHA_CALLS), mha_key, FRONT_VERIFIED),
    }


def _record(hsv, monkeypatch, run, frame=True):
    """Keys of every conv / activation / CUDA-core conv / attention launch (through the launch record) and of every
    frame-op call (through the ops wrappers) during ``run``."""
    from megatts2_hierspeechpp_b200 import _lib
    from test_gpu_frame_variants import KEYERS, call_key
    ops = hsv.ops
    ops.set_umma_debug(0)
    ops.set_act_variant(0)
    ops.set_mha_variant(0)
    fams = _families(ops)
    seen = {f: {} for f in list(fams) + ["frame"]}
    last = {f: ops.last_launch_config(f)["launches"] for f in fams}
    orig = _lib.check

    def recording_check(rc, what):
        orig(rc, what)
        for f, (calls, key, _) in fams.items():
            if what in calls:
                c = ops.last_launch_config(f)
                if c["launches"] != last[f]:        # empty calls launch nothing
                    last[f] = c["launches"]
                    k = key(c)
                    seen[f][k] = seen[f].get(k, 0) + 1

    def wrap(name, fn):
        def rec(*args, **kwargs):
            k = call_key(fn, name, args, kwargs)
            seen["frame"][k] = seen["frame"].get(k, 0) + 1
            return fn(*args, **kwargs)
        return rec

    origs = {n: getattr(ops, n) for n in KEYERS} if frame else {}
    monkeypatch.setattr(_lib, "check", recording_check)
    for n, fn in origs.items():
        monkeypatch.setattr(ops, n, wrap(n, fn))
    try:
        with torch.no_grad():
            run()
        torch.cuda.synchronize()
    finally:
        monkeypatch.setattr(_lib, "check", orig)
        for n, fn in origs.items():
            monkeypatch.setattr(ops, n, fn)
    return seen


def _assert_census(hsv, name, seen, need=("conv", "act", "direct")):
    from test_gpu_frame_variants import FRAME_VERIFIED
    ops = hsv.ops
    fams = _families(ops)
    names = {ops.LAUNCH_CONV: "conv", ops.LAUNCH_ACT: "act", ops.LAUNCH_DIRECT: "direct", ops.LAUNCH_MHA: "attention",
             "frame": "frame"}
    bad = {}
    for f, keys in seen.items():
        print(f"\n[census] {name} {names[f]}: " + (", ".join(f"{k} x{n}" for k, n in sorted(keys.items())) or "none"),
              end="")
        verified = FRAME_VERIFIED if f == "frame" else fams[f][2]
        if set(keys) - verified:
            bad[names[f]] = sorted(set(keys) - verified)
        if names[f] in need:
            assert keys, f"{name}: no {names[f]} launch recorded"
    print()
    assert not bad, f"{name} launches variants no case verifies: {bad}"


def _bench_model(workload, batch):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    import bench
    wl = bench.make_workload(argparse.Namespace(workload=workload, batch=batch, seconds=10.0), 0)
    return wl, bench.build_model(wl, DEV)


SR_CENSUS = [("speechsr24", 1), ("speechsr24", 16), ("chain24", 1), ("speechsr48", 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("workload,batch", SR_CENSUS, ids=[f"{w}-B{b}" for w, b in SR_CENSUS])
def test_census_sr_workloads_verified(hsv, monkeypatch, workload, batch):
    """One eager forward of a SpeechSR benchmark workload (bench.py's model and inputs, 10 s)."""
    wl, model = _bench_model(workload, batch)
    seen = _record(hsv, monkeypatch, lambda: model(*[t.to(DEV) for t in wl["host_inputs"]]))
    _assert_census(hsv, wl["name"], seen)


def _lens(lens):
    return torch.tensor(lens, dtype=torch.int32, device=DEV)


@functools.lru_cache(maxsize=None)
def _sr_model(which):
    import megatts2_hierspeechpp_b200 as hsv
    from conftest import golden_sd
    m = (hsv.SpeechSR24 if which == 24 else hsv.SpeechSR48)(100, 40, **hsv.SR_CFG)
    m.load_state_dict(golden_sd(f"speechsr{which}_state.npz"), strict=True)
    return m.to(DEV).eval()


@pytest.mark.gpu
def test_census_ragged_speechsr24_verified(hsv, monkeypatch):
    sr = _sr_model(24)
    lens = [32000, 2, 7, 16001, 3334]
    x = torch.randn(len(lens), 1, max(lens), generator=torch.Generator().manual_seed(24)) * 0.3
    seen = _record(hsv, monkeypatch, lambda: sr(x.to(DEV), lengths=_lens(lens)))
    _assert_census(hsv, f"ragged SpeechSR24 B={len(lens)}", seen)


@pytest.mark.gpu
def test_census_ragged_batches_conv_act_verified(hsv, monkeypatch):
    """The ragged vocoder, SpeechSR48 and text-to-vec tail batches (their CUDA-core conv and frame-op launches are
    censused by the direct / frame files; recorded here too)."""
    from oracle import synth
    voc = hsv.Vocoder()
    voc.load_state_dict(synth.vocoder_sd(1234), strict=True)
    voc.to(DEV).eval()
    lens = [500, 1, 2, 37, 499, 250]
    z, g = synth.vocoder_inputs(len(lens), max(lens), seed=21)
    _assert_census(hsv, f"ragged vocoder B={len(lens)}",
                   _record(hsv, monkeypatch, lambda: voc(z.to(DEV), g.to(DEV), lengths=_lens(lens))))
    sr = _sr_model(48)
    lens = [48000, 1, 7, 16001, 3333]
    x = torch.randn(len(lens), 1, max(lens), generator=torch.Generator().manual_seed(48)) * 0.3
    _assert_census(hsv, f"ragged SpeechSR48 B={len(lens)}",
                   _record(hsv, monkeypatch, lambda: sr(x.to(DEV), lengths=_lens(lens))))
    tail = hsv.TTVTail()
    tail.load_state_dict(synth.ttv_tail_sd(3456), strict=True)
    tail.to(DEV).eval()
    lens = [333, 300, 129, 1, 2]
    z, _, g = synth.ttv_tail_inputs(len(lens), max(lens), seed=22)
    _assert_census(hsv, f"ragged text-to-vec tail B={len(lens)}",
                   _record(hsv, monkeypatch, lambda: tail(z.to(DEV), None, g.to(DEV), lengths=_lens(lens))),
                   need=("conv",))


@pytest.mark.gpu
def test_census_per_item_synthesizer_conv_act_verified(hsv, monkeypatch):
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
    seen = None
    for ids, Tp, Tmp in batches:
        B = len(ids)
        src, f0 = torch.zeros(B, 1024, Tp), torch.zeros(B, 1, 4 * Tp)
        mel = torch.zeros(2 * B, 80, Tmp)
        for j, i in enumerate(ids):
            T, Tm = lengths[i], prompts[i]
            src[j, :, :T], f0[j, :, :4 * T] = ins[i][0][0], ins[i][1][0]
            mel[j, :, :Tm], mel[B + j, :, :Tm] = ins[i][2][0], ins[i][2][1]
        vl, tl = _lens([lengths[i] for i in ids]), _lens([prompts[i] for i in ids] * 2)
        s = _record(hsv, monkeypatch, lambda: model.voice_conversion_noise_control(
            src.to(DEV), vl, mel.to(DEV), tl, f0.to(DEV), 0.333, False, 0.3, per_item=True))
        if seen is None:
            seen = s
        else:
            for f, keys in s.items():
                for k, c in keys.items():
                    seen[f][k] = seen[f].get(k, 0) + c
    _assert_census(hsv, f"per-item synthesizer B={n} ({len(batches)} batches)", seen)


STREAM_CENSUS = [(24, 4, 320), (24, 256, 320), (48, 4, 320), (48, 256, 320)]


@pytest.mark.gpu
@pytest.mark.parametrize("which,S,N", STREAM_CENSUS, ids=[f"{w}k-S{s}-N{n}" for w, s, n in STREAM_CENSUS])
def test_census_speechsr_stream_verified(hsv, monkeypatch, which, S, N):
    """Eager steps of SpeechSRStream: streams starting, continuing with short and full chunks, ending, and idle
    slots (the windows of valid length 0 in every ragged launch)."""
    st = hsv.SpeechSRStream(_sr_model(which), S, N)
    gen = torch.Generator().manual_seed(S)
    z = torch.zeros(S, dtype=torch.int32)
    plan = []
    for step in range(5):
        n, s, e = z.clone(), z.clone(), z.clone()
        for b in range(S):
            if b % 3 == 2:
                continue                                    # idle slot
            if step == 0:
                s[b] = 1
            n[b] = N if (b + step) % 2 else 2 * ((b * 37 + step * 11) % (N // 2))
            e[b] = int(step == 3 and b % 3 == 1)
        if step == 4:
            n.zero_(), s.zero_(), e.zero_()                   # an all-idle step
        plan.append((torch.randn(S, N, generator=gen) * 0.3, n, s, e))

    def run():
        for x, n, s, e in plan:
            st(x.to(DEV), n.to(DEV), s.to(DEV), e.to(DEV))

    seen = _record(hsv, monkeypatch, run)
    _assert_census(hsv, f"SpeechSRStream {which} kHz S={S} N={N}", seen)
