"""Variable-length vocoder job on one GPU: today's equal-length schedule vs the ragged (``lengths=``) schedule.

    python tools/bench_ragged.py [--utts 256] [--tmin 100] [--tmax 1000] [--max-batch 16] [--frame-multiple 50]
                                 [--parallel-blocks 1]

The job: ``--utts`` utterances with T uniform in [tmin, tmax] frames (torch generator seeded 1111), utterance i's
z / g from ``synthetic.vocoder_inputs(1, T_i, seed=1111 + i)``, vocoder weights ``synthetic.vocoder_sd(1234)``.

(a) ``runtime.bucket_by_length`` micro-batches through ``CudaGraphRunner(capture_after=2)``, the setting INTEGRATION.md
    recommends for variable lengths.  The timed pass uses a fresh runner, as a stream of one-off lengths would see it:
    nothing is captured, every micro-batch runs eagerly (the untimed pass loads modules and folds weights).
(b) ``runtime.ragged_batches`` micro-batches (padded to a multiple of ``--frame-multiple`` frames) with ``lengths=``
    through one ``CudaGraphRunner``; the untimed pass captures one graph per padded shape, the timed pass replays.

Each schedule runs once untimed, then ``--reps`` timed passes of the whole job (CUDA events, final synchronise; batch
inputs are assembled on the device before timing, per-utterance outputs are sliced and cloned inside it).  Every
utterance's waveform is compared between (a) and (b) with ``torch.equal``.  Prints one JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import megatts2_hierspeechpp_b200 as hsv  # noqa: E402
from megatts2_hierspeechpp_b200 import synthetic  # noqa: E402
from megatts2_hierspeechpp_b200.runtime import CudaGraphRunner, bucket_by_length, ragged_batches  # noqa: E402

HOP, SR = 320, 16000


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except Exception:   # the number is reported beside the results; a missing nvidia-smi must not stop the run
        return None


def timed(run, reps):
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        outs = run()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return ms, outs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=256)
    ap.add_argument("--tmin", type=int, default=100)
    ap.add_argument("--tmax", type=int, default=1000)
    ap.add_argument("--max-batch", type=int, default=16)
    ap.add_argument("--frame-multiple", type=int, default=50)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--parallel-blocks", type=int, default=1, help="multi-stream resblocks (bench.py's default: 1)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ragged.py needs a CUDA device")
    dev = torch.device("cuda:0")

    lengths = torch.randint(args.tmin, args.tmax + 1, (args.utts,), generator=torch.Generator().manual_seed(1111)).tolist()
    ins = [synthetic.vocoder_inputs(1, T, seed=1111 + i) for i, T in enumerate(lengths)]
    z = [a.to(dev) for a, _ in ins]
    g = [b.to(dev) for _, b in ins]
    voc = hsv.Vocoder()
    voc.load_state_dict(synthetic.vocoder_sd(1234), strict=True)
    voc.to(dev).eval()
    voc.dec.parallel_blocks = voc.sn.parallel_blocks = bool(args.parallel_blocks)

    # (a) equal-length micro-batches
    buckets = bucket_by_length(range(args.utts), lengths, args.max_batch)
    a_in = [(torch.cat([z[i] for i in ids]), torch.cat([g[i] for i in ids])) for ids in buckets]

    def run_a(runner):
        res = {}
        for ids, (zb, gb) in zip(buckets, a_in):
            w = runner(zb, gb)
            for j, i in enumerate(ids):
                res[i] = w[j].clone()
        return res

    # (b) ragged micro-batches
    batches = ragged_batches(range(args.utts), lengths, args.max_batch, args.frame_multiple)
    b_in = []
    for ids, Tp in batches:
        zb = torch.zeros(len(ids), z[0].shape[1], Tp, device=dev)
        for j, i in enumerate(ids):
            zb[j, :, :lengths[i]] = z[i][0]
        b_in.append((zb, torch.cat([g[i] for i in ids]),
                     torch.tensor([lengths[i] for i in ids], dtype=torch.int32, device=dev)))
    runner_b = CudaGraphRunner(voc)

    def run_b():
        res = {}
        for (ids, _), (zb, gb, ln) in zip(batches, b_in):
            w = runner_b(zb, gb, ln)
            for j, i in enumerate(ids):
                res[i] = w[j, :, :lengths[i] * HOP].clone()
        return res

    with torch.no_grad():
        run_a(CudaGraphRunner(voc, capture_after=2))           # untimed
        torch.cuda.synchronize()
        runners_a = []                                           # one fresh runner per timed pass

        def fresh_a():
            runners_a.append(CudaGraphRunner(voc, capture_after=2))
            return run_a(runners_a[-1])

        ms_a, out_a = timed(fresh_a, args.reps)
        cap_a_timed = sum(r.captures for r in runners_a)
        run_b()                                                  # untimed: captures
        torch.cuda.synchronize()
        cap_b0 = runner_b.captures
        ms_b, out_b = timed(run_b, args.reps)
        cap_b_timed = runner_b.captures - cap_b0
        tails_zero = True
        for (ids, _), (zb, gb, ln) in zip(batches, b_in):
            w = runner_b(zb, gb, ln)
            tails_zero &= all(bool((w[j, :, lengths[i] * HOP:] == 0).all()) for j, i in enumerate(ids))

    mismatches = sum(0 if torch.equal(out_a[i], out_b[i]) else 1 for i in range(args.utts))
    audio_s = sum(lengths) * HOP / SR
    padded = sum(len(ids) * Tp for ids, Tp in batches)

    def summary(ms):
        med = statistics.median(ms)
        return {"ms_per_job": round(med, 2), "ms_all": [round(m, 2) for m in ms],
                "audio_s_per_s": round(audio_s / (med / 1e3), 1)}

    line = {
        "tool": "bench_ragged",
        "device": torch.cuda.get_device_name(0),
        "power_limit_w": power_limit_w(),
        "job": {"utterances": args.utts, "frames": [args.tmin, args.tmax], "seed": 1111, "audio_s": round(audio_s, 2),
                "distinct_lengths": len(set(lengths)), "max_batch": args.max_batch,
                "parallel_blocks": bool(args.parallel_blocks)},
        "a_bucket_by_length": {**summary(ms_a), "micro_batches": len(buckets), "captures_timed": cap_a_timed,
                               "padded_frame_fraction": 0.0},
        "b_ragged": {**summary(ms_b), "micro_batches": len(batches), "frame_multiple": args.frame_multiple,
                     "graph_shapes": len({(len(ids), Tp) for ids, Tp in batches}), "graphs_captured": runner_b.captures,
                     "captures_timed": cap_b_timed, "padded_frame_fraction": round(1 - sum(lengths) / padded, 4),
                     "tails_zero": tails_zero},
        "speedup_b_over_a": round(statistics.median(ms_a) / statistics.median(ms_b), 3),
        "mismatches": mismatches,
    }
    print(json.dumps(line), flush=True)
    if mismatches or cap_b_timed or not tails_zero:
        sys.exit(1)


if __name__ == "__main__":
    main()
