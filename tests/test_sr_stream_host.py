"""Streaming SpeechSR on the host: the lookahead / halo derivation, the host mirror of the schedule and argument checks
(no GPU)."""
import ctypes
import random

import pytest
import torch

from conftest import golden_sd
from oracle import functional as OF

from megatts2_hierspeechpp_b200 import SR_CFG, SpeechSR24, SpeechSR48, ops
from megatts2_hierspeechpp_b200.sr_stream import (MAX_STREAM_OUTPUT, SRStreamSchedule, SpeechSRStream, _act_reach,
                                                  history_len, stream_reach)


def _model(which):
    return (SpeechSR24 if which == 24 else SpeechSR48)(100, 40, **SR_CFG)


def test_activation_reach_from_its_filters():
    # 12-tap x2 up-sample (replicate pad 5) then 12-tap x2 low-pass: output t reads x[t - 5, t + 5]
    assert _act_reach(_model(48).dec.activation_post) == (5, 5)


@pytest.mark.parametrize("which, R, H", [(48, 115, 77), (24, 107, 144)])
def test_reach_from_layer_list(which, R, H):
    gen = _model(which).dec
    # post: widest resblock (k 11, d 1/3/5: 3 x (5 + 5d + 5 + 5)) + activation_post 5 + conv_post 3 = 98 per side;
    # interpolation + conv_pre: ceil(ratio * 5.5 + 0.5) output samples
    assert stream_reach(gen) == (R, R)
    assert history_len(R, R, ops.SR_RATIOS[gen.scale]) == H
    assert H % ops.SR_RATIOS[gen.scale][1] == 0


@pytest.mark.parametrize("which", [24, 48])
def test_reach_bounds_the_oracle(which):
    """Perturbing the input from sample n on leaves outputs below ratio * n - lookahead unchanged, and perturbing it
    before sample m leaves outputs from ratio * m + halo on unchanged (the oracle of the reference's forward, in fp64).
    (The bounds are not tight in floating point: the farthest contributions are products of the filters' smallest taps
    and round away.)"""
    sd = {k: v.double() for k, v in golden_sd(f"speechsr{which}_state.npz").items()}
    R, HL = stream_reach(_model(which).dec)
    r = 3 if which == 48 else 1.5
    L = 600
    gen = torch.Generator().manual_seed(5)
    x = torch.randn(1, 1, L, generator=gen, dtype=torch.float64) * 0.3
    y = OF.speechsr(sd, x, which)[0, 0]
    for n in (200, 402):
        xp = x.clone()
        xp[..., n:] += torch.randn(L - n, generator=gen, dtype=torch.float64)
        first = int(((OF.speechsr(sd, xp, which)[0, 0] - y).abs() > 0).nonzero().min())
        assert int(r * n) - R <= first < int(r * n)
    for m in (200, 402):
        xp = x.clone()
        xp[..., :m] += torch.randn(m, generator=gen, dtype=torch.float64)
        last = int(((OF.speechsr(sd, xp, which)[0, 0] - y).abs() > 0).nonzero().max())
        assert int(r * m) <= last < int(r * m) + HL


def _stream_model(sched_args):
    """Independent model of a stream's output count: after every step, min(total, max(0, ratio * received - R)) are
    out before the end, all of them at the end."""
    ratio, R, steps = sched_args
    up, down = ratio
    out, recv = [], 0
    for i, n in enumerate(steps):
        recv += n
        last = i == len(steps) - 1
        out.append(recv * up // down if last else max(0, recv * up // down - R))
    return [b - a for a, b in zip([0] + out[:-1], out)]


@pytest.mark.parametrize("ratio", [(3, 1), (3, 2)])
def test_schedule_mirror_random_streams(ratio):
    """Random chunkings, starts, ends, idle steps and slot reuse: every slot's n_out sequence per stream equals the
    independent count, a stream's outputs sum to its offline length, and never run ahead of received * ratio - R."""
    up, down = ratio
    S, N, R = 6, 40, 115 if ratio == (3, 1) else 107
    rng = random.Random(7)
    sch = SRStreamSchedule(S, N, ratio, R)
    cur = [None] * S          # per slot: list of n_new of the open stream, and its n_out so far
    done = 0
    for _ in range(600):
        n_new, start, end = [0] * S, [False] * S, [False] * S
        for b in range(S):
            u = rng.random()
            if cur[b] is None:
                if u < 0.3:
                    start[b] = True
                    n_new[b] = rng.randrange(0, N + 1, down)
                    end[b] = rng.random() < 0.1
            elif u < 0.2:
                continue        # idle
            else:
                n_new[b] = rng.randrange(0, N + 1, down)
                end[b] = rng.random() < 0.08
        n_out = sch.step(n_new, start, end)
        for b in range(S):
            if start[b]:
                cur[b] = ([], [])
            if cur[b] is None:
                assert n_out[b] == 0
                continue
            if n_new[b] or end[b] or start[b]:
                cur[b][0].append(n_new[b])
            else:
                assert n_out[b] == 0
                continue
            cur[b][1].append(n_out[b])
            recv = sum(cur[b][0])
            if not end[b]:
                assert sum(cur[b][1]) <= max(0, recv * up // down - R)
            if end[b]:
                assert cur[b][1] == _stream_model((ratio, R, cur[b][0]))
                assert sum(cur[b][1]) == recv * up // down
                cur[b] = None
                done += 1
    assert done > 50


def test_schedule_rejects_what_the_device_would_ignore():
    sch = SRStreamSchedule(3, 320, (3, 2), 107)
    with pytest.raises(ValueError, match="odd"):
        sch.step([3, 0, 0], [True, False, False], [False] * 3)
    with pytest.raises(ValueError, match="outside"):
        sch.step([322, 0, 0], [True, False, False], [False] * 3)
    with pytest.raises(ValueError, match="no open stream"):
        sch.step([0, 0, 0], [False] * 3, [True, False, False])
    with pytest.raises(ValueError, match="no open stream"):
        sch.step([0, 2, 0], [False] * 3, [False] * 3)
    with pytest.raises(ValueError, match="entries"):
        sch.step([0, 0], [False] * 2, [False] * 2)
    assert sch.received == [0, 0, 0] and sch.open == [False] * 3     # a rejected step changes nothing
    assert sch.step([320, 0, 0], [True, False, False], [False] * 3) == [480 - 107, 0, 0]
    assert sch.step([0, 0, 0], [False] * 3, [True, False, False]) == [107, 0, 0]   # an end with n_new = 0 flushes
    sch48 = SRStreamSchedule(1, 4, (3, 1), 115)
    assert sch48.step([3], [True], [False]) == [0]                   # odd lengths are fine at 48 kHz
    sch48.received[0] = MAX_STREAM_OUTPUT // 3 - 2
    with pytest.raises(ValueError, match="2\\^24"):
        sch48.step([4], [False], [False])


def test_ops_and_stream_reject_cpu_and_wrong_dtypes():
    x = torch.zeros(2, 1, 16)
    w = torch.zeros(4, 1, 7)
    vl = torch.zeros(2, dtype=torch.int32)
    org = torch.zeros(2, 3, dtype=torch.int64)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.sr_pre_interp_stream(x, w, None, 48, (vl, vl), org, (3, 1))
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.sr_stream_window(torch.zeros(2, 8), vl, vl, vl, torch.zeros(2, 4), torch.zeros(2, 3, dtype=torch.int64),
                             (3, 1), 10)
    with pytest.raises(ValueError, match="ratio"):
        ops._req_ratio((2, 1))
    with pytest.raises(RuntimeError, match="CUDA"):
        SpeechSRStream(_model(48), 2, 320)
    with pytest.raises(TypeError):
        SpeechSRStream(torch.nn.Linear(2, 2), 2, 320)


def test_stream_entry_points_check_arguments():
    from megatts2_hierspeechpp_b200 import _lib, build
    build.build()
    lib = _lib.load()
    one = ctypes.c_void_p(16)
    rc = lib.hsv_sr_pre_interp_stream(one, one, None, one, one, None, one, 1, 8, 16, 48, 3, 1, None)
    assert rc == -1 and b"null" in lib.hsv_last_error()
    rc = lib.hsv_sr_pre_interp_stream(one, one, None, one, one, one, one, 1, 8, 16, 48, 2, 1, None)
    assert rc == -1 and b"ratio" in lib.hsv_last_error()
    args = [one] * 11
    rc = lib.hsv_sr_stream_window(*args, 2, 320, 143, 3, 2, 107, None)
    assert rc == -1 and b"multiple" in lib.hsv_last_error()
    rc = lib.hsv_sr_stream_emit(*([one] * 8), 2, 77, 77, 1200, 1075, None)
    assert rc == -1 and b"bad shape" in lib.hsv_last_error()
